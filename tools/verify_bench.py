"""Throughput of the device signature / id checks: prints one JSON line.

- the card's name and power limit;
- sw_verify events/s at batch sizes 4096, 65 536 and 1 M for M = 64 and M = 1024 members: device time (engine CUDA
  events around the call: its copies and the kernel), kernel time alone (torch.profiler), and host wall time of the
  whole call.  One warm-up call per shape; the L2 is flushed (sw_flush_l2) before every timed call;
- sw_ingest_verified against sw_ingest on the same signed gossip batch (1 M events by default);
- libsodium (PyNaCl) verifications per second on one host core, measured in the same run.

Signed events are 65 536 distinct pickled events (swirld.py's Event layout) signed with seeded keys, tiled.

    python tools/verify_bench.py [--reps R] [--ingest-n N]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import pickle
import subprocess
import sys
import time
from collections import namedtuple

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "py-swirld_b200"))
Event = namedtuple("Event", "d p t c s")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                                   # (the query is informative only)
        return {"name": "unknown", "error": str(exc)}


def offsets(chunks):
    off = np.zeros(len(chunks) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in chunks])
    return off


def signed_batch(nacl, M, distinct=65536, total=1 << 20):
    keys = [nacl.crypto_sign_seed_keypair(hashlib.sha256(b"bench%d" % i).digest()) for i in range(M)]
    rng = np.random.default_rng(1)
    creator = rng.integers(0, M, distinct).astype(np.int32)
    msgs, wires, sigs = [], [], np.empty((distinct, 64), np.uint8)
    for i in range(distinct):
        c = int(creator[i])
        p = (hashlib.blake2b(b"p0%d" % i, digest_size=32).digest(), hashlib.blake2b(b"p1%d" % i, digest_size=32).digest())
        msg = pickle.dumps((b"payload %d" % i, p, 1.7e9 + i, keys[c][0]))
        s = nacl.crypto_sign(msg, keys[c][1])[:64]
        msgs.append(msg)
        wires.append(pickle.dumps(Event(b"payload %d" % i, p, 1.7e9 + i, keys[c][0], s)))
        sigs[i] = np.frombuffer(s, np.uint8)
    ids = np.stack([np.frombuffer(hashlib.blake2b(w, digest_size=32).digest(), np.uint8) for w in wires])
    T = total // distinct
    mo, wo = offsets(msgs), offsets(wires)
    tile = lambda o: np.append((o[:-1][None, :] + o[-1] * np.arange(T)[:, None]).ravel(), o[-1] * T)
    return {"pks": [k[0] for k in keys], "creator": np.tile(creator, T), "sig": np.tile(sigs, (T, 1)),
            "msg": np.tile(np.frombuffer(b"".join(msgs), np.uint8), T), "msg_off": tile(mo),
            "ids": np.tile(ids, (T, 1)), "wire": np.tile(np.frombuffer(b"".join(wires), np.uint8), T), "wire_off": tile(wo),
            "one": (msgs, sigs, creator, keys)}


def sliced(b, n):
    mo, wo = b["msg_off"], b["wire_off"]
    return (b["creator"][:n], b["sig"][:n], b["msg"][:mo[n]], mo[:n + 1], b["ids"][:n], b["wire"][:wo[n]], wo[:n + 1])


def kernel_ms(fn):
    """Device time of the k_verify launches of fn(), from torch.profiler (None when it records none)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        us = 0.0
        for ev in prof.events():
            if "k_verify" in ev.name and "keys" not in ev.name and "table" not in ev.name:
                us += getattr(ev, "device_time", None) or getattr(ev, "cuda_time", 0.0)
        return us / 1e3 if us > 0 else None
    except Exception:
        return None


def bench_verify(engine, b, M, reps):
    e = engine.Engine(M, 16)
    assert e.set_member_keys(b["pks"]) == 0
    out = {}
    for n in (4096, 65536, 1 << 20):
        args = sliced(b, n)
        st = e.verify(*args)                                   # warm-up (and correctness: every event valid)
        assert int((st == 3).sum()) == n, "verify rejected valid events"
        dev, wall = [], []
        for _ in range(reps if n >= 65536 else 4 * reps):
            e.flush_l2(256 << 20)
            e.record(0)
            t0 = time.perf_counter()
            e.verify(*args)
            wall.append(time.perf_counter() - t0)
            e.record(1)
            dev.append(e.elapsed_ms(0, 1))
        kms = kernel_ms(lambda: e.verify(*args))
        out[str(n)] = {"device_ms": float(np.median(dev)), "wall_ms": 1e3 * float(np.median(wall)),
                       "kernel_ms": kms,
                       "device_ev_per_s": n / (np.median(dev) / 1e3), "wall_ev_per_s": n / float(np.median(wall)),
                       "kernel_ev_per_s": (n / (kms / 1e3)) if kms else None,
                       "h2d_bytes": int(args[2].size + args[5].size + 100 * n)}
    e.close()
    return out


def bench_ingest(engine, nacl, M, N):
    from swirld_b200 import traces
    tr = traces.gossip(M, N, 5)
    keys = [nacl.crypto_sign_seed_keypair(hashlib.sha256(b"ingest%d" % i).digest()) for i in range(M)]
    items, hs = [], []
    for i in range(tr.N):
        c = int(tr.creator[i])
        p = () if tr.p0[i] < 0 else (hs[tr.p0[i]], hs[tr.p1[i]])
        d, t = b"tx%d" % i, float(tr.t[i])
        ev = Event(d, p, t, keys[c][0], nacl.crypto_sign(pickle.dumps((d, p, t, keys[c][0])), keys[c][1])[:64])
        hs.append(hashlib.blake2b(pickle.dumps(ev), digest_size=32).digest())
        items.append((hs[-1], ev))
    t0 = time.perf_counter()
    cols = engine.event_columns(items, {k[0]: i for i, k in enumerate(keys)})
    columns_s = time.perf_counter() - t0
    perm = np.random.default_rng(2).permutation(N)
    c = {k: (v[perm] if k not in ("msg", "msg_off", "wire", "wire_off") else v) for k, v in cols.items()}
    ms = [cols["msg"][cols["msg_off"][i]:cols["msg_off"][i + 1]].tobytes() for i in perm]
    ws = [cols["wire"][cols["wire_off"][i]:cols["wire_off"][i + 1]].tobytes() for i in perm]
    msg, mo = np.frombuffer(b"".join(ms), np.uint8), offsets(ms)
    wire, wo = np.frombuffer(b"".join(ws), np.uint8), offsets(ws)
    res = {"events": N, "members": M, "event_columns_s": columns_s}
    for rep in range(2):                                       # (the second round is the one reported)
        e = engine.Engine(M, N + 8)
        e.set_member_keys([k[0] for k in keys])
        t0 = time.perf_counter()
        _, m1 = e.ingest(c["ids"], c["p0_ids"], c["p1_ids"], c["creator"], c["t"], c["sig"])
        e.sync()
        t_plain = time.perf_counter() - t0
        e2 = engine.Engine(M, N + 8)
        e2.set_member_keys([k[0] for k in keys])
        t0 = time.perf_counter()
        _, m2 = e2.ingest_verified(c["ids"], c["p0_ids"], c["p1_ids"], c["creator"], c["t"], c["sig"], msg, mo, wire, wo)
        e2.sync()
        t_ver = time.perf_counter() - t0
        assert m1 == N and m2 == N
        res.update({"ingest_s": t_plain, "ingest_verified_s": t_ver, "ingest_ev_per_s": N / t_plain,
                    "ingest_verified_ev_per_s": N / t_ver})
        e.close(); e2.close()
    return res


def libsodium_rate(nacl, b, n=20000):
    msgs, sigs, creator, keys = b["one"]
    t0 = time.perf_counter()
    for i in range(n):
        nacl.crypto_sign_open(sigs[i].tobytes() + msgs[i], keys[creator[i]][0])
    return n / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ingest-n", type=int, default=1 << 20)
    a = ap.parse_args()
    from nacl import bindings as nacl
    from swirld_b200 import engine
    res = {"card": card()}
    for M in (64, 1024):
        b = signed_batch(nacl, M)
        res["verify_M%d" % M] = bench_verify(engine, b, M, a.reps)
        if M == 64:
            res["libsodium_verify_per_s_one_core"] = libsodium_rate(nacl, b)
    res["ingest_M64"] = bench_ingest(engine, nacl, 64, a.ingest_n)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
