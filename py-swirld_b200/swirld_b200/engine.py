"""ctypes binding of libswirld_b200.so (include/swirld_b200.h).

There is no CPU implementation behind this module: if the CUDA library is not
built, or no CUDA device is present, construction raises.  The oracle under
oracle/ is test infrastructure and is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libswirld_b200.so")
PEER_HANDLE_BYTES = 128          # SW_PEER_HANDLE_BYTES

SW_E = {-1: "SW_E_ARG", -2: "SW_E_INDEX", -3: "SW_E_KEY", -4: "SW_E_CUDA", -5: "SW_E_CAPACITY",
        -6: "SW_E_PARENT", -7: "SW_E_FORK", -8: "SW_E_UNSUPPORTED"}

# every symbol include/swirld_b200.h declares (tests check the library exports them all)
SYMBOLS = [
    "sw_create", "sw_destroy", "sw_reset", "sw_rewind", "sw_event_record", "sw_event_elapsed_ms", "sw_last_error", "sw_append", "sw_divide_rounds",
    "sw_decide_fame", "sw_find_order", "sw_n_events", "sw_n_divided", "sw_max_round",
    "sw_n_transactions", "sw_get_round", "sw_get_witness_flags", "sw_get_famous", "sw_get_can_see",
    "sw_get_witness_table", "sw_get_consensus", "sw_get_transactions", "sw_get_idx", "sw_get_height",
    "sw_sync", "sw_stats", "sw_flush_l2", "sw_version", "sw_debug_counters", "sw_peer_handle", "sw_peer_connect",
    "sw_save", "sw_load", "sw_members", "sw_ingest", "sw_lookup", "sw_batch_divide_rounds",
    "sw_set_member_keys", "sw_verify", "sw_ingest_verified",
]


class SwStats(C.Structure):
    _fields_ = [("ms_divide_rounds", C.c_double), ("ms_decide_fame", C.c_double),
                ("ms_find_order", C.c_double), ("ms_can_see", C.c_double),
                ("kernel_launches", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("events", C.c_int64), ("events_divided", C.c_int64), ("ms_rounds_kernel", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s (%d): %s" % (SW_E.get(code, "SW_E_?"), code, msg))
        self.code = code


_lib = None


def load_library(path: str = LIB_PATH):
    """dlopen the CUDA library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise RuntimeError(
            "%s is missing: build it with `python -m swirld_b200.build` (nvcc, sm_100a). "
            "This engine has no CPU fallback." % path)
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    P = C.POINTER
    L.sw_create.argtypes = [i32, i32, P(C.c_int64), i32, i32, P(vp)]
    L.sw_destroy.argtypes = [vp]; L.sw_destroy.restype = None
    L.sw_reset.argtypes = [vp]
    L.sw_rewind.argtypes = [vp]
    L.sw_event_record.argtypes = [vp, i32]
    L.sw_event_elapsed_ms.argtypes = [vp, i32, i32, P(C.c_double)]
    L.sw_last_error.argtypes = [vp]; L.sw_last_error.restype = C.c_char_p
    L.sw_append.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.sw_divide_rounds.argtypes = [vp, i32, i32]
    L.sw_decide_fame.argtypes = [vp, vp, i32]
    L.sw_find_order.argtypes = [vp, vp, i32]
    for f in ("sw_n_events", "sw_n_divided", "sw_max_round", "sw_n_transactions", "sw_sync"):
        getattr(L, f).argtypes = [vp]
    for f in ("sw_get_round", "sw_get_witness_flags", "sw_get_famous", "sw_get_can_see",
              "sw_get_witness_table", "sw_get_transactions", "sw_get_idx", "sw_get_height"):
        getattr(L, f).argtypes = [vp, i32, i32, vp]
    L.sw_get_consensus.argtypes = [vp, vp, i32]
    L.sw_stats.argtypes = [vp, P(SwStats)]
    L.sw_flush_l2.argtypes = [vp, i64]
    L.sw_version.argtypes = []
    L.sw_debug_counters.argtypes = [vp, vp, i32]
    L.sw_peer_handle.argtypes = [vp, vp]
    L.sw_peer_connect.argtypes = [vp, i32, i32, vp]
    L.sw_members.argtypes = [vp]
    L.sw_ingest.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.sw_lookup.argtypes = [vp, i32, vp, vp]
    L.sw_set_member_keys.argtypes = [vp, vp]
    L.sw_verify.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.sw_ingest_verified.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.sw_batch_divide_rounds.argtypes = [vp, i32, vp, vp]
    L.sw_save.argtypes = [vp, C.c_char_p]
    L.sw_load.argtypes = [C.c_char_p, i32, i32, P(vp)]
    _lib = L
    return L


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _bytes_col(buf, off, n):
    buf = np.ascontiguousarray(np.frombuffer(buf, np.uint8) if isinstance(buf, (bytes, bytearray)) else buf, np.uint8)
    off = np.ascontiguousarray(off, np.int64)
    assert off.shape[0] == n + 1 and off[0] >= 0 and off[-1] <= buf.size
    if buf.size == 0:
        buf = np.zeros(1, np.uint8)
    return buf, off


def event_columns(events, member_of):
    """The columns sw_ingest_verified / sw_verify read, from (id, Event) pairs (Event = the reference's namedtuple
    (d, p, t, c, s)) and a public key -> member index map.  The signed bytes and the hashed bytes are serialised
    exactly as the reference does (swirld.py:95, 99): pickle.dumps(ev[:-1]) and pickle.dumps(ev).  A creator not in
    the map gets member -1, so its signature never verifies."""
    import pickle
    n = len(events)
    zero = bytes(32)
    ids = np.empty((n, 32), np.uint8); p0 = np.zeros((n, 32), np.uint8); p1 = np.zeros((n, 32), np.uint8)
    creator = np.empty(n, np.int32); t = np.empty(n, np.float64); sig = np.zeros((n, 64), np.uint8)
    msgs, wires = [], []
    for i, (h, ev) in enumerate(events):
        ids[i] = np.frombuffer(h, np.uint8)
        if ev.p:
            p0[i] = np.frombuffer(ev.p[0] or zero, np.uint8)
            p1[i] = np.frombuffer(ev.p[1] or zero, np.uint8)
        s = bytes(ev.s)
        creator[i] = member_of.get(ev.c, -1) if len(s) == 64 else -1     # (a signature of another length never verifies)
        t[i] = ev.t
        sig[i, :min(64, len(s))] = np.frombuffer(s[:64], np.uint8)
        msgs.append(pickle.dumps(ev[:-1]))
        wires.append(pickle.dumps(ev))
    msg_off = np.zeros(n + 1, np.int64); msg_off[1:] = np.cumsum([len(m) for m in msgs])
    wire_off = np.zeros(n + 1, np.int64); wire_off[1:] = np.cumsum([len(w) for w in wires])
    return {"ids": ids, "p0_ids": p0, "p1_ids": p1, "creator": creator, "t": t, "sig": sig,
            "msg": np.frombuffer(b"".join(msgs), np.uint8), "msg_off": msg_off,
            "wire": np.frombuffer(b"".join(wires), np.uint8), "wire_off": wire_off}


class Engine:
    """One node-view of the hashgraph on one GPU; thin, index-space."""

    def __init__(self, M: int, capacity: int, stake=None, coin_period: int = 6, device: int = 0):
        self._lib = load_library()
        self.M, self.capacity = int(M), int(capacity)
        h = C.c_void_p()
        st = None
        if stake is not None:
            arr = (C.c_int64 * M)(*[int(s) for s in stake])
            st = C.cast(arr, C.POINTER(C.c_int64))
        rc = self._lib.sw_create(M, capacity, st, coin_period, device, C.byref(h))
        if rc < 0:
            raise EngineError(rc, (self._lib.sw_last_error(None) or b"").decode())
        self._h = h

    # -- checkpoint / resume
    def save(self, path: str):
        self._chk(self._lib.sw_save(self._h, os.fsencode(path)))

    @classmethod
    def load(cls, path: str, device: int = 0, capacity: int = 0) -> "Engine":
        lib = load_library()
        h = C.c_void_p()
        rc = lib.sw_load(os.fsencode(path), device, capacity, C.byref(h))
        if rc < 0:
            raise EngineError(rc, (lib.sw_last_error(None) or b"").decode())
        self = cls.__new__(cls)
        self._lib, self._h = lib, h
        self.M = self._chk(lib.sw_members(h))
        self.capacity = capacity
        return self

    # -- life cycle
    def close(self):
        if getattr(self, "_h", None):
            self._lib.sw_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc < 0:
            msg = (self._lib.sw_last_error(self._h) or b"").decode()
            if rc == -2:
                raise IndexError(msg)
            if rc == -3:
                raise KeyError(msg)
            raise EngineError(rc, msg)
        return rc

    def reset(self):
        self._chk(self._lib.sw_reset(self._h))

    def rewind(self):
        self._chk(self._lib.sw_rewind(self._h))

    def record(self, slot):
        self._chk(self._lib.sw_event_record(self._h, slot))

    def elapsed_ms(self, a, b):
        ms = C.c_double()
        self._chk(self._lib.sw_event_elapsed_ms(self._h, a, b, C.byref(ms)))
        return ms.value

    # -- the path
    def append(self, p0, p1, creator, t, sig):
        p0 = np.ascontiguousarray(p0, np.int32); p1 = np.ascontiguousarray(p1, np.int32)
        creator = np.ascontiguousarray(creator, np.int32); t = np.ascontiguousarray(t, np.float64)
        sig = np.ascontiguousarray(sig, np.uint8)
        n = p0.shape[0]
        assert p1.shape[0] == n and creator.shape[0] == n and t.shape[0] == n and sig.size == 64 * n
        self._chk(self._lib.sw_append(self._h, n, _ptr(p0), _ptr(p1), _ptr(creator), _ptr(t), _ptr(sig)))

    def ingest(self, ids, p0_ids, p1_ids, creator, t, sig):
        """sw_ingest: events named by 32-byte ids (parents by id, zeros = none), any order; returns the arrival index
        of every input event (-1 = rejected) and the number appended."""
        ids = np.ascontiguousarray(ids, np.uint8).reshape(-1, 32)
        n = ids.shape[0]
        p0_ids = np.ascontiguousarray(p0_ids, np.uint8).reshape(n, 32)
        p1_ids = np.ascontiguousarray(p1_ids, np.uint8).reshape(n, 32)
        creator = np.ascontiguousarray(creator, np.int32); t = np.ascontiguousarray(t, np.float64)
        sig = np.ascontiguousarray(sig, np.uint8).reshape(n, 64)
        out = np.empty(n, np.int32)
        m = self._chk(self._lib.sw_ingest(self._h, n, _ptr(ids), _ptr(p0_ids), _ptr(p1_ids), _ptr(creator), _ptr(t), _ptr(sig), _ptr(out)))
        return out, m

    # -- is_valid_event's crypto checks on the GPU (Ed25519 signature, BLAKE2b id)
    def set_member_keys(self, pks) -> int:
        """The members' 32-byte public keys in member order; returns how many of them libsodium would reject."""
        pk = np.ascontiguousarray(np.frombuffer(b"".join(bytes(k) for k in pks), np.uint8)
                                  if not isinstance(pks, np.ndarray) else pks, np.uint8).reshape(-1, 32)
        assert pk.shape[0] == self.M
        return self._chk(self._lib.sw_set_member_keys(self._h, _ptr(pk)))

    def verify(self, creator, sig, msg, msg_off, ids, wire, wire_off):
        """sw_verify: per event, bit 0 = the signature verifies, bit 1 = the id is BLAKE2b-256 of the wire bytes."""
        creator = np.ascontiguousarray(creator, np.int32)
        n = creator.shape[0]
        sig = np.ascontiguousarray(sig, np.uint8).reshape(n, 64)
        ids = np.ascontiguousarray(ids, np.uint8).reshape(n, 32)
        msg, msg_off = _bytes_col(msg, msg_off, n)
        wire, wire_off = _bytes_col(wire, wire_off, n)
        out = np.zeros(n, np.uint8)
        self._chk(self._lib.sw_verify(self._h, n, _ptr(creator), _ptr(sig), _ptr(msg), _ptr(msg_off), _ptr(ids),
                                      _ptr(wire), _ptr(wire_off), _ptr(out)))
        return out

    def ingest_verified(self, ids, p0_ids, p1_ids, creator, t, sig, msg, msg_off, wire, wire_off):
        """sw_ingest_verified: ingest() that first checks the new events' signatures and ids; returns (index, appended)."""
        ids = np.ascontiguousarray(ids, np.uint8).reshape(-1, 32)
        n = ids.shape[0]
        p0_ids = np.ascontiguousarray(p0_ids, np.uint8).reshape(n, 32)
        p1_ids = np.ascontiguousarray(p1_ids, np.uint8).reshape(n, 32)
        creator = np.ascontiguousarray(creator, np.int32); t = np.ascontiguousarray(t, np.float64)
        sig = np.ascontiguousarray(sig, np.uint8).reshape(n, 64)
        msg, msg_off = _bytes_col(msg, msg_off, n)
        wire, wire_off = _bytes_col(wire, wire_off, n)
        out = np.empty(n, np.int32)
        m = self._chk(self._lib.sw_ingest_verified(self._h, n, _ptr(ids), _ptr(p0_ids), _ptr(p1_ids), _ptr(creator),
                                                   _ptr(t), _ptr(sig), _ptr(msg), _ptr(msg_off), _ptr(wire),
                                                   _ptr(wire_off), _ptr(out)))
        return out, m

    def lookup(self, ids):
        ids = np.ascontiguousarray(ids, np.uint8).reshape(-1, 32)
        out = np.empty(ids.shape[0], np.int32)
        self._chk(self._lib.sw_lookup(self._h, ids.shape[0], _ptr(ids), _ptr(out)))
        return out

    def append_trace(self, tr, first=0, n=None):
        n = tr.N - first if n is None else n
        s = slice(first, first + n)
        self.append(tr.p0[s], tr.p1[s], tr.creator[s], tr.t[s], tr.sig[s])

    def divide_rounds(self, first, n):
        self._chk(self._lib.sw_divide_rounds(self._h, first, n))

    def decide_fame(self):
        cap = max(64, self.n_divided + 2)
        if getattr(self, "_newc_buf", None) is None or self._newc_buf.size < cap:
            self._newc_buf = np.empty(cap, np.int32)
        n = self._chk(self._lib.sw_decide_fame(self._h, _ptr(self._newc_buf), self._newc_buf.size))
        return self._newc_buf[:n].tolist()

    def find_order(self, new_c):
        a = np.ascontiguousarray(sorted(new_c), np.int32)
        if a.size == 0:
            return 0
        return self._chk(self._lib.sw_find_order(self._h, _ptr(a), a.size))

    # -- views
    @property
    def n_events(self):
        return self._lib.sw_n_events(self._h)

    @property
    def n_divided(self):
        return self._lib.sw_n_divided(self._h)

    @property
    def n_transactions(self):
        return self._lib.sw_n_transactions(self._h)

    @property
    def max_round(self):
        return self._chk(self._lib.sw_max_round(self._h))

    def _get(self, fn, dtype, first, n, width=1):
        out = np.empty((n, width) if width > 1 else n, dtype)
        if n:
            self._chk(fn(self._h, first, n, _ptr(out)))
        return out

    def rounds(self, first=0, n=None):
        return self._get(self._lib.sw_get_round, np.int32, first, self.n_divided - first if n is None else n)

    def witness_flags(self, first=0, n=None):
        return self._get(self._lib.sw_get_witness_flags, np.uint8, first, self.n_divided - first if n is None else n)

    def famous(self, first=0, n=None):
        return self._get(self._lib.sw_get_famous, np.int8, first, self.n_events - first if n is None else n)

    def can_see(self, first=0, n=None):
        n = self.n_divided - first if n is None else n
        out = np.empty((n, self.M), np.int32)
        if n:
            self._chk(self._lib.sw_get_can_see(self._h, first, n, _ptr(out)))
        return out

    def witness_table(self, first_round=0, n_rounds=None):
        n_rounds = self.max_round + 1 - first_round if n_rounds is None else n_rounds
        out = np.empty((n_rounds, self.M), np.int32)
        if n_rounds:
            self._chk(self._lib.sw_get_witness_table(self._h, first_round, n_rounds, _ptr(out)))
        return out

    def consensus(self):
        buf = np.empty(max(1, self.max_round + 2), np.int32)
        n = self._chk(self._lib.sw_get_consensus(self._h, _ptr(buf), buf.size))
        return buf[:n].copy()

    def transactions(self, first=0, n=None):
        return self._get(self._lib.sw_get_transactions, np.int32, first, self.n_transactions - first if n is None else n)

    def idx(self, first=0, n=None):
        return self._get(self._lib.sw_get_idx, np.int32, first, self.n_events - first if n is None else n)

    def heights(self, first=0, n=None):
        return self._get(self._lib.sw_get_height, np.int32, first, self.n_events - first if n is None else n)

    def sync(self):
        self._chk(self._lib.sw_sync(self._h))

    def stats(self):
        s = SwStats()
        self._chk(self._lib.sw_stats(self._h, C.byref(s)))
        return s.as_dict()

    def debug_counters(self, clear=True):
        out = np.zeros(16, np.int64)
        self._chk(self._lib.sw_debug_counters(self._h, _ptr(out), 1 if clear else 0))
        return out

    # -- several GPUs of one box, M > 64 (include/swirld_b200.h: sw_peer_handle / sw_peer_connect)
    def peer_handle(self) -> bytes:
        """The CUDA IPC handles (PEER_HANDLE_BYTES bytes) of this engine's exchange buffer and can_see table."""
        buf = C.create_string_buffer(PEER_HANDLE_BYTES)
        self._chk(self._lib.sw_peer_handle(self._h, C.cast(buf, C.c_void_p)))
        return buf.raw

    def peer_connect(self, rank: int, nranks: int, handles: bytes):
        """handles = the nranks handles concatenated in rank order; call before the first divide_rounds."""
        assert len(handles) == PEER_HANDLE_BYTES * nranks
        buf = C.create_string_buffer(handles, len(handles))
        self._chk(self._lib.sw_peer_connect(self._h, rank, nranks, C.cast(buf, C.c_void_p)))

    def flush_l2(self, nbytes=256 << 20):
        self._chk(self._lib.sw_flush_l2(self._h, nbytes))

    def results(self):
        """Same dict as oracle.Oracle.results() (index space)."""
        return {"round": self.rounds(), "witness": self.witness_flags(),
                "witness_table": self.witness_table(), "famous": self.famous(),
                "consensus": self.consensus(), "transactions": self.transactions()}


def batch_divide_rounds(engines, firsts, counts):
    """sw_batch_divide_rounds: divide_rounds of several independent node-views (M <= 64) in one call."""
    B = len(engines)
    arr = (C.c_void_p * B)(*[e._h for e in engines])
    f = np.ascontiguousarray(firsts, np.int32)
    n = np.ascontiguousarray(counts, np.int32)
    engines[0]._chk(engines[0]._lib.sw_batch_divide_rounds(C.cast(arr, C.c_void_p), B, _ptr(f), _ptr(n)))


def run_engine(tr, K, stake=None, coin_period=6, device=0, find_order=True):
    """Feed a trace with the call schedule K; returns results() + new_c per call."""
    from .traces import chunks
    e = Engine(tr.M, tr.N, stake, coin_period, device)
    ncs = []
    for first, cnt in chunks(tr.N, K):
        e.append_trace(tr, first, cnt)
        e.divide_rounds(first, cnt)
        nc = e.decide_fame()
        if find_order:
            e.find_order(nc)
        ncs.append(sorted(nc))
    res = e.results()
    res["new_c_per_call"] = ncs
    res["can_see"] = e.can_see()
    res["stats"] = e.stats()
    res["engine"] = e
    return res
