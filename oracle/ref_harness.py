"""Tier-0 oracle: drive the UNMODIFIED reference (swirld.py of Lapin0t/py-swirld)
through its own hot-path methods on an index-space trace.

TEST INFRASTRUCTURE ONLY.  Works only where the environment variable
SWIRLD_REFERENCE names a checkout of the reference; used by
`oracle/make_golden.py` to produce the fixtures under `tests/golden/` (which the
tests compare against) and by bench.py's optional timing of the reference.
Nothing is copied from the reference: it is imported from where it lies,
behind the `pysodium` shim in `oracle/pysodium_shim/`.

Recipe (SURVEY.md Appendix A.2): one `Node`, the state its constructor made for
its own root event thrown away, events fed with integer ids through
`add_event`, then one (`divide_rounds`, `decide_fame`, `find_order`) triple per
chunk of K events -- the call schedule of `Node.main` (swirld.py:324-328).
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import time
from collections import defaultdict

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("SWIRLD_REFERENCE", "")


def reference_available() -> bool:
    return bool(REF) and os.path.isfile(os.path.join(REF, "swirld.py"))


def load_reference():
    """Import the reference module unmodified (shim first on sys.path)."""
    shim = os.path.join(HERE, "pysodium_shim")
    if shim not in sys.path:
        sys.path.insert(0, shim)
    if REF not in sys.path:
        sys.path.insert(1, REF)
    import swirld  # noqa: the reference, from SWIRLD_REFERENCE
    return swirld


def run_reference(tr, K: int, stake=None, snapshots: bool = False):
    """Feed trace `tr` (swirld_b200.traces.Trace) to the reference in chunks of
    K events (K may also be an explicit list of chunk sizes).  Returns a dict of numpy arrays in index space plus timings.

    famous: int8[N]  -1 = no entry in Node.famous, 0 = False, 1 = True
    witness: uint8[N] 1 iff the event is a value of Node.witnesses[r] for some r
    """
    swirld = load_reference()
    M, N = tr.M, tr.N
    stake = {c: 1 for c in range(M)} if stake is None else dict(enumerate(stake))
    from pysodium import crypto_sign_keypair
    with contextlib.redirect_stdout(io.StringIO()):
        nd = swirld.Node(crypto_sign_keypair(), {}, M, stake)
    # throw away what the ctor registered for its own root (swirld.py:75-80)
    nd.hg = {}
    nd.head = None
    nd.round = {}
    nd.tbd = set()
    nd.height = {}
    nd.can_see = {}
    nd.witnesses = defaultdict(dict)
    nd.transactions = []
    nd.idx = {}

    p0, p1, cr = tr.p0.tolist(), tr.p1.tolist(), tr.creator.tolist()
    tt = tr.t.tolist()
    sig = [bytes(tr.sig[i]) for i in range(N)]
    t_dr = t_df = t_fo = 0.0
    new_c_per_call = []
    snaps = []
    sink = io.StringIO()
    first = 0
    sizes = iter(K) if isinstance(K, (list, tuple)) else None
    while first < N:
        cnt = min(next(sizes) if sizes is not None else K, N - first)
        ids = list(range(first, first + cnt))
        for i in ids:
            par = () if p0[i] < 0 else (p0[i], p1[i])
            nd.add_event(i, swirld.Event(None, par, tt[i], cr[i], sig[i]))
        with contextlib.redirect_stdout(sink):
            a = time.perf_counter()
            nd.divide_rounds(ids)
            b = time.perf_counter()
            new_c = nd.decide_fame()
            c = time.perf_counter()
            nd.find_order(new_c)
            d = time.perf_counter()
        sink.seek(0)
        sink.truncate(0)
        t_dr += b - a
        t_df += c - b
        t_fo += d - c
        new_c_per_call.append(sorted(new_c))
        if snapshots:
            snaps.append(_extract(nd, first + cnt, M))
        first += cnt
    out = _extract(nd, N, M)
    out["can_see_node"] = nd
    out["new_c_per_call"] = new_c_per_call
    out["t_divide_rounds"] = t_dr
    out["t_decide_fame"] = t_df
    out["t_find_order"] = t_fo
    if snapshots:
        out["snapshots"] = snaps
    return out


def _extract(nd, n, M):
    rnd = np.full(n, -1, dtype=np.int32)
    for h, r in nd.round.items():
        rnd[h] = r
    wit = np.zeros(n, dtype=np.uint8)
    max_r = max(nd.witnesses) if nd.witnesses else -1
    wtab = np.full((max_r + 1, M), -1, dtype=np.int32)
    for r, d in nd.witnesses.items():
        for c, h in d.items():
            wit[h] = 1
            wtab[r, c] = h
    fam = np.full(n, -1, dtype=np.int8)
    for h, v in nd.famous.items():
        fam[h] = 1 if v else 0
    return {
        "round": rnd,
        "witness": wit,
        "witness_table": wtab,
        "famous": fam,
        "consensus": np.array(sorted(nd.consensus), dtype=np.int32),
        "transactions": np.array(nd.transactions, dtype=np.int32),
    }


def can_see_matrix(nd, n, M) -> np.ndarray:
    """Node.can_see (dict of dicts) as an int32[n, M] matrix, -1 = absent."""
    out = np.full((n, M), -1, dtype=np.int32)
    for h, row in nd.can_see.items():
        for c, k in row.items():
            out[h, c] = k
    return out
