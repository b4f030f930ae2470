"""The device signature / id checks (sw_set_member_keys, sw_verify, sw_ingest_verified) against libsodium's verdicts:
the pinned vectors bit for bit, a 1 M-event batch with known corruptions, and a signed gossip trace ingested in
shuffled batches (accepted set, consensus) against a CPU replay of is_valid_event."""
import hashlib
import os
import pickle
import random
from collections import namedtuple

import numpy as np
import pytest

import oracle as orc
from util import assert_same

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURE = os.path.join(ROOT, "tests", "golden", "ed25519_vectors.npz")
Event = namedtuple("Event", "d p t c s")


def _blake(b):
    return np.frombuffer(hashlib.blake2b(b, digest_size=32).digest(), np.uint8)


def _offsets(chunks):
    off = np.zeros(len(chunks) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in chunks])
    return off


# ---------------------------------------------------------------- (a) pinned vectors
def test_pinned_vectors_bit_for_bit():
    from swirld_b200 import engine
    z = np.load(FIXTURE)
    n = z["verdict"].size
    # every distinct key is a member; engines of at most 1024 members
    keys, member = [], np.empty(n, np.int32)
    index = {}
    for i in range(n):
        k = z["pk"][i].tobytes()
        if k not in index:
            index[k] = len(keys)
            keys.append(k)
        member[i] = index[k]
    key_ok = {z["pk"][i].tobytes(): int(z["key_ok"][i]) for i in range(n)}
    for g0 in range(0, len(keys), 1024):
        gkeys = keys[g0:g0 + 1024]
        e = engine.Engine(len(gkeys), 16)
        bad = e.set_member_keys(gkeys)
        assert bad == sum(1 - key_ok[k] for k in gkeys)
        sel = np.nonzero((member >= g0) & (member < g0 + len(gkeys)))[0]
        msgs = [z["msg"][z["msg_off"][i]:z["msg_off"][i + 1]].tobytes() for i in sel]
        ids = z["msg_digest"][sel].copy()
        wrong = np.arange(sel.size) % 3 == 1                   # every third id does not match its wire bytes
        ids[wrong, 5] ^= 0x40
        msg, off = np.frombuffer(b"".join(msgs) or b"\0", np.uint8), _offsets(msgs)
        st = e.verify(member[sel] - g0, z["sig"][sel], msg, off, ids, msg, off)
        want = z["verdict"][sel] | (2 * (~wrong)).astype(np.uint8)
        bad_at = np.nonzero(st != want)[0]
        assert bad_at.size == 0, [(str(z["kind_names"][z["kind"][sel[i]]]), int(st[i]), int(want[i])) for i in bad_at[:10]]
        assert e.verify(member[sel] - g0, z["sig"][sel], msg, off, ids, msg, off).tolist() == st.tolist()
        e.close()
    # BLAKE2b across the block boundaries and 1 MiB (creator -1: bit 0 is 0)
    e = engine.Engine(1, 16)
    e.set_member_keys([keys[0]])
    nb = z["blake_digest"].shape[0]
    ids = z["blake_digest"].copy()
    ids[1::2, 31] ^= 1
    st = e.verify(np.full(nb, -1, np.int32), np.zeros((nb, 64), np.uint8), np.zeros(1, np.uint8), np.zeros(nb + 1, np.int64),
                  ids, z["blake_in"], z["blake_off"])
    assert st.tolist() == [2 if i % 2 == 0 else 0 for i in range(nb)]


# ---------------------------------------------------------------- (b) a 1 M-event batch
def _signed_events(nkeys, ndistinct, seed):
    b = pytest.importorskip("nacl.bindings")
    rng = random.Random(seed)
    keys = [b.crypto_sign_seed_keypair(hashlib.sha256(b"key%d:%d" % (seed, i)).digest()) for i in range(nkeys)]
    creator = np.array([rng.randrange(nkeys) for _ in range(ndistinct)], np.int32)
    msgs, wires, sigs = [], [], np.empty((ndistinct, 64), np.uint8)
    for i in range(ndistinct):
        msg = pickle.dumps((None, (), float(i), keys[creator[i]][0]))
        sig = b.crypto_sign(msg, keys[creator[i]][1])[:64]
        msgs.append(msg)
        wires.append(pickle.dumps((None, (), float(i), keys[creator[i]][0], sig)))
        sigs[i] = np.frombuffer(sig, np.uint8)
    return [k[0] for k in keys], creator, sigs, msgs, wires


def test_large_batch_exact_status():
    from swirld_b200 import engine
    pks, creator, sigs, msgs, wires = _signed_events(64, 65536, 11)
    D, T = len(msgs), 16
    N = D * T
    ids = np.stack([_blake(w) for w in wires])
    msg1, moff1 = np.frombuffer(b"".join(msgs), np.uint8), _offsets(msgs)
    wire1, woff1 = np.frombuffer(b"".join(wires), np.uint8), _offsets(wires)
    tile = lambda o, T: (o[:-1][None, :] + o[-1] * np.arange(T)[:, None]).ravel()
    msg, moff = np.tile(msg1, T).copy(), np.append(tile(moff1, T), moff1[-1] * T)
    wire, woff = np.tile(wire1, T).copy(), np.append(tile(woff1, T), woff1[-1] * T)
    cr, sg, idc = np.tile(creator, T), np.tile(sigs, (T, 1)), np.tile(ids, (T, 1))
    want = np.full(N, 3, np.uint8)
    rng = np.random.default_rng(3)
    pick = rng.choice(N, 4000, replace=False)
    for j, i in enumerate(pick):
        kind = j % 5
        if kind == 0:
            sg[i, rng.integers(64)] ^= 1 << int(rng.integers(8)); want[i] = 2
        elif kind == 1:
            msg[moff[i] + rng.integers(moff[i + 1] - moff[i])] ^= 1; want[i] = 2
        elif kind == 2:
            idc[i, rng.integers(32)] ^= 0x80; want[i] = 1
        elif kind == 3:
            wire[woff[i] + rng.integers(woff[i + 1] - woff[i])] ^= 4; want[i] = 1
        else:
            cr[i] = (cr[i] + 1) % 64; want[i] = 2
    e = engine.Engine(64, 16)
    assert e.set_member_keys(pks) == 0
    st = e.verify(cr, sg, msg, moff, idc, wire, woff)
    assert np.array_equal(st, want), np.nonzero(st != want)[0][:20]
    s = e.stats()
    assert s["kernel_launches"] >= 3 and s["h2d_bytes"] >= msg.size + wire.size and s["d2h_bytes"] >= N


# ---------------------------------------------------------------- (c) a signed gossip trace, ingested with the checks
def _signed_trace(M, N, seed, tamper):
    """traces.gossip's graph with real events: Event(d, p, t, c, s) signed over dumps(ev[:-1]), id = BLAKE2b(dumps(ev)).
    tamper: {event: kind} -- 0 bad signature bytes, 1 payload changed after signing, 2 signed with another member's
    key; the id is that of the tampered event, so its descendants name it and hang below it."""
    b = pytest.importorskip("nacl.bindings")
    from swirld_b200 import traces
    tr = traces.gossip(M, N, seed)
    keys = [b.crypto_sign_seed_keypair(hashlib.sha256(b"member%d" % i).digest()) for i in range(M)]
    evs, hs = [], []
    for i in range(tr.N):
        c = int(tr.creator[i])
        p = () if tr.p0[i] < 0 else (hs[tr.p0[i]], hs[tr.p1[i]])
        d = b"tx%d" % i
        t = float(tr.t[i])
        signer = keys[(c + 1) % M][1] if tamper.get(i) == 2 else keys[c][1]
        s = b.crypto_sign(pickle.dumps((d, p, t, keys[c][0])), signer)[:64]
        if tamper.get(i) == 0:
            s = s[:40] + bytes([s[40] ^ 0x10]) + s[41:]
        ev = Event(d if tamper.get(i) != 1 else b"forged", p, t, keys[c][0], s)
        evs.append(ev)
        hs.append(hashlib.blake2b(pickle.dumps(ev), digest_size=32).digest())
    return tr, [k[0] for k in keys], list(zip(hs, evs))


def _is_valid_event_crypto(h, ev):
    """The reference's two crypto checks (swirld.py:97-103), with libsodium."""
    b = pytest.importorskip("nacl.bindings")
    try:
        b.crypto_sign_open(ev.s + pickle.dumps(ev[:-1]), ev.c)
    except Exception:
        return False
    return hashlib.blake2b(pickle.dumps(ev), digest_size=32).digest() == h


def test_signed_gossip_trace_ingested_with_checks():
    from swirld_b200 import engine
    from swirld_b200.traces import Trace, chunks
    M, N = 16, 20000
    tamper = {19000: 0, 19250: 1, 19500: 2, 19800: 0, 19990: 1}
    tr, pks, items = _signed_trace(M, N, 21, tamper)
    member = {pk: i for i, pk in enumerate(pks)}
    # CPU replay: toposort + is_valid_event + the fork rule.  The graph is fork-free and every batch holds only events
    # whose parents arrived before or in it, so an event is accepted iff it and all its ancestors pass the crypto checks.
    ok = np.zeros(N, bool)
    for i, (h, ev) in enumerate(items):
        par = [] if tr.p0[i] < 0 else [tr.p0[i], tr.p1[i]]
        ok[i] = _is_valid_event_crypto(h, ev) and all(ok[q] for q in par)
    assert (~ok).sum() > len(tamper) and ok[:19000].all()
    cols = engine.event_columns(items, member)
    e = engine.Engine(M, N + 8)
    assert e.set_member_keys(pks) == 0
    plain = engine.Engine(M, N + 8)
    rng = np.random.default_rng(5)
    arrival = np.full(N, -1, np.int64)
    first = 0
    sizes = [16, 1, 7, 500, 3, 2473, 3000, 4000, 4000, 3000, 2000, 1000]
    assert sum(sizes) == N
    take = lambda a, idx: a[idx]
    for cnt in sizes:
        batch = rng.permutation(np.arange(first, first + cnt))
        if first:
            batch = np.concatenate([batch, rng.integers(0, first, 2)])      # + two events sent before
        ms = [cols["msg"][cols["msg_off"][i]:cols["msg_off"][i + 1]].tobytes() for i in batch]
        ws = [cols["wire"][cols["wire_off"][i]:cols["wire_off"][i + 1]].tobytes() for i in batch]
        args = [take(cols[k], batch) for k in ("ids", "p0_ids", "p1_ids", "creator", "t", "sig")]
        out, m = e.ingest_verified(*args, np.frombuffer(b"".join(ms), np.uint8), _offsets(ms),
                                   np.frombuffer(b"".join(ws), np.uint8), _offsets(ws))
        new = batch[:cnt]
        assert m == int(ok[new].sum())
        assert np.array_equal(out[:cnt] >= 0, ok[new])
        arrival[new[out[:cnt] >= 0]] = out[:cnt][out[:cnt] >= 0]
        if first:
            assert np.array_equal(out[cnt:], arrival[batch[cnt:]])
        _, m2 = plain.ingest(*args)
        assert m2 == cnt                                       # without the checks the tampered events get in
        first += cnt
    assert e.n_events == int(ok.sum()) and plain.n_events == N
    assert np.array_equal(np.sort(arrival[ok]), np.arange(int(ok.sum())))
    # consensus on the verified graph == the oracle on the same arrival order
    order = np.argsort(np.where(ok, arrival, N + np.arange(N)))[:int(ok.sum())]
    remap = lambda p: np.where(p >= 0, arrival[np.maximum(p, 0)], -1).astype(np.int32)
    tr2 = Trace(M, remap(tr.p0[order]), remap(tr.p1[order]), tr.creator[order], tr.t[order], cols["sig"][order], "verified")
    K = 1500
    o = orc.run_oracle(tr2, K)
    ncs = []
    for f0, c in chunks(tr2.N, K):
        e.divide_rounds(f0, c)
        nc = e.decide_fame()
        e.find_order(nc)
        ncs.append(sorted(nc))
    r = e.results()
    r["new_c_per_call"] = ncs
    assert_same(o, r, what="graph ingested with the crypto checks")


# ---------------------------------------------------------------- (d) the API contract
def test_verify_api_contract():
    from swirld_b200 import engine
    b = pytest.importorskip("nacl.bindings")
    M = 1024
    keys = [b.crypto_sign_seed_keypair(hashlib.sha256(b"big%d" % i).digest()) for i in range(M)]
    e = engine.Engine(M, 64)
    msgs = [b"event %d" % i for i in range(3000)]
    creator = np.array([(i * 37) % M for i in range(3000)], np.int32)
    sig = np.stack([np.frombuffer(b.crypto_sign(msgs[i], keys[creator[i]][1])[:64], np.uint8) for i in range(3000)])
    ids = np.stack([_blake(x) for x in msgs])
    msg, off = np.frombuffer(b"".join(msgs), np.uint8), _offsets(msgs)
    with pytest.raises(engine.EngineError) as ei:
        e.verify(creator, sig, msg, off, ids, msg, off)
    assert ei.value.code == -1
    pks = [k[0] for k in keys]
    pks[5] = bytes(32)                                         # a small-order key (order 4): member 5 never verifies
    pks[6] = b"\xff" * 31 + b"\x7f"                            # y >= p
    assert e.set_member_keys(pks) == 2
    want = np.where(np.isin(creator, [5, 6]), 2, 3).astype(np.uint8)
    assert np.array_equal(e.verify(creator, sig, msg, off, ids, msg, off), want)
    cr = creator.copy(); cr[:3] = [-1, M, M + 7]
    assert e.verify(cr, sig, msg, off, ids, msg, off)[:3].tolist() == [2, 2, 2]
    e.reset()
    assert np.array_equal(e.verify(creator, sig, msg, off, ids, msg, off), want)
    e.rewind()
    assert np.array_equal(e.verify(creator, sig, msg, off, ids, msg, off), want)
    # the verify changed no engine state
    assert e.n_events == 0
