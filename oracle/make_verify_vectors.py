"""Pinned Ed25519 / BLAKE2b vectors for the device checks of sw_verify (tests/golden/ed25519_vectors.npz).

Deterministic: keys come from crypto_sign_seed_keypair with fixed seeds, messages from fixed byte patterns, and the
edge cases (small-order and mixed-order keys, non-canonical encodings) from the pure-Python model in
tests/ed25519_model.py.  Every signature vector records libsodium's verdict (through PyNaCl) and the BLAKE2b-256 of
its message, so the GPU test needs neither PyNaCl nor its version.

    python oracle/make_verify_vectors.py [out.npz]     (default: tests/golden/ed25519_vectors.npz)
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ed25519_model as m  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ed25519_vectors.npz")
LENGTHS = [0, 1, 47, 48, 63, 64, 175, 176, 1000]      # R || A adds 64: every SHA-512 padding boundary
BLAKE_LENGTHS = [0, 1, 127, 128, 129, 255, 256, 257, 1 << 20]
MIB = 1 << 20


def pattern(n: int, salt: int) -> bytes:
    """n message bytes; periodic so that the 1 MiB vectors compress."""
    block = hashlib.sha512(b"msg%d" % salt).digest() * 4
    return (block * (n // len(block) + 1))[:n]


def libsodium_verdict(sig: bytes, msg: bytes, pk: bytes) -> bool:
    from nacl import bindings as b
    from nacl.exceptions import CryptoError
    try:
        b.crypto_sign_open(sig + msg, pk)
        return True
    except (CryptoError, ValueError):
        return False


def key(i: int):
    """(pk, a, prefix) of crypto_sign_seed_keypair(bytes([i]) * 32)."""
    return m.seed_keypair(bytes([i]) * 32)


def enc_y(y: int, sign: int) -> bytes:
    return (y | (sign << 255)).to_bytes(32, "little")


def off_curve_ys(count: int, start: int = 2):
    out, y = [], start
    while len(out) < count:
        if m.point_from_y(y) is None:
            out.append(y)
        y += 1
    return out


def build():
    vec = []                                                    # (kind, pk, sig, msg)

    def add(kind, pk, sig, msg):
        vec.append((kind, bytes(pk), bytes(sig), bytes(msg)))

    keys = [key(i) for i in range(8)]
    # valid signatures, across the SHA-512 padding boundaries, plus 1 MiB
    for n in LENGTHS:
        pk, a, pre = keys[0]
        msg = pattern(n, n)
        add("valid", pk, m.sign_with(a, pre, pk, msg), msg)
    for i in range(1, 8):
        pk, a, pre = keys[i]
        msg = pattern(100 + 37 * i, i)
        add("valid", pk, m.sign_with(a, pre, pk, msg), msg)
    pk, a, pre = keys[0]
    big = pattern(MIB, 99)
    add("valid", pk, m.sign_with(a, pre, pk, big), big)
    # single-bit flips in R, s, msg and pk
    pk, a, pre = keys[1]
    msg = pattern(120, 7)
    sig = m.sign_with(a, pre, pk, msg)
    for bit in (0, 1, 100, 254, 255):
        s = bytearray(sig); s[bit // 8] ^= 1 << (bit % 8); add("flip_R", pk, s, msg)
    for bit in (0, 1, 100, 252, 255):
        s = bytearray(sig); s[32 + bit // 8] ^= 1 << (bit % 8); add("flip_s", pk, s, msg)
    for bit in (0, 7, 500, 959):
        mm = bytearray(msg); mm[bit // 8] ^= 1 << (bit % 8); add("flip_msg", pk, sig, mm)
    for bit in (0, 1, 128, 254, 255):
        kk = bytearray(pk); kk[bit // 8] ^= 1 << (bit % 8); add("flip_pk", kk, sig, msg)
    # s + L, s with the top bits set
    s_int = int.from_bytes(sig[32:], "little")
    add("s_plus_L", pk, sig[:32] + (s_int + m.L).to_bytes(32, "little"), msg)
    for top in (0x10, 0x20, 0x80, 0xF0, 0xE0):
        s = bytearray(sig); s[63] |= top; add("s_top_bits", pk, s, msg)
    # every blocklisted encoding as R and as A, both sign bits
    pk2, a2, pre2 = keys[2]
    msg2 = pattern(64, 2)
    sig2 = m.sign_with(a2, pre2, pk2, msg2)
    for y in m.BLOCKLIST_YS:
        for sign in (0, 1):
            e = enc_y(y, sign)
            add("small_order_R", pk2, e + sig2[32:], msg2)
            add("small_order_A", e, sig2, msg2)
    # R = identity with the cofactorless equation holding (s = k a), and A = R = identity, s = 0
    ident = enc_y(1, 0)
    k = m.challenge(ident, pk2, msg2)
    add("identity_R_equation_holds", pk2, ident + (k * a2 % m.L).to_bytes(32, "little"), msg2)
    add("identity_A_identity_R_s0", ident, ident + bytes(32), msg2)
    # A with y >= p: all 19 values, both signs
    for y in range(m.P, 2 ** 255):
        for sign in (0, 1):
            add("A_y_ge_p", enc_y(y, sign), sig2, msg2)
    # A and R not on the curve
    for y in off_curve_ys(3):
        for sign in (0, 1):
            add("A_off_curve", enc_y(y, sign), sig2, msg2)
            add("R_off_curve", pk2, enc_y(y, sign) + sig2[32:], msg2)
    # mixed-order A = [a]B + T (T of order 2, 4 or 8): the cofactorless equation holds iff [k]T = 0
    pk3, a3, pre3 = keys[3]
    A3 = m.decode(pk3)
    for ti, T in enumerate(m.small_order_points()):
        if m.encode(T) == ident:
            continue
        Amix = m.encode(m.add(A3, T))
        found = {0: 0, 1: 0}
        ctr = 0
        while min(found.values()) < 1:
            msg = pattern(80, 1000 * ti + ctr)
            ctr += 1
            sig = m.sign_with(a3, pre3, Amix, msg)
            kk = m.challenge(sig[:32], Amix, msg)
            cls = 0 if kk % 8 == 0 else 1
            if found[cls] < 1:
                found[cls] += 1
                add("mixed_order_A_k0mod8" if cls == 0 else "mixed_order_A_k_not0mod8", Amix, sig, msg)
    # canonical R vs non-canonical R: y in [0, 19) against y + p, both signs, over a valid s
    pk4, a4, pre4 = keys[4]
    msg4 = pattern(90, 4)
    sig4 = m.sign_with(a4, pre4, pk4, msg4)
    for y in range(19):
        for sign in (0, 1):
            add("R_canonical_small_y", pk4, enc_y(y, sign) + sig4[32:], msg4)
            add("R_noncanonical_y", pk4, enc_y(y + m.P, sign) + sig4[32:], msg4)
    # the canonical R of the signature with its y + p twin does not exist (y_R >= 19): the pair then is
    # (valid R, R with the sign bit flipped)
    add("R_sign_flipped", pk4, bytes(sig4[:31]) + bytes([sig4[31] ^ 0x80]) + sig4[32:], msg4)

    kinds = sorted(set(v[0] for v in vec))
    verdict = np.array([libsodium_verdict(s, msg, pk) for _, pk, s, msg in vec], np.uint8)
    model = np.array([m.verify(s, msg, pk) for _, pk, s, msg in vec], np.uint8)
    assert np.array_equal(verdict, model), "the model disagrees with libsodium: %s" % [
        vec[i][0] for i in np.nonzero(verdict != model)[0]]
    msgs = [v[3] for v in vec]
    msg_off = np.zeros(len(vec) + 1, np.int64)
    msg_off[1:] = np.cumsum([len(x) for x in msgs])
    blake_in = [pattern(n, 5000 + n) for n in BLAKE_LENGTHS]
    blake_off = np.zeros(len(blake_in) + 1, np.int64)
    blake_off[1:] = np.cumsum([len(x) for x in blake_in])
    return {
        "kind": np.array([kinds.index(v[0]) for v in vec], np.int32),
        "kind_names": np.array(kinds),
        "pk": np.frombuffer(b"".join(v[1] for v in vec), np.uint8).reshape(-1, 32),
        "sig": np.frombuffer(b"".join(v[2] for v in vec), np.uint8).reshape(-1, 64),
        "msg": np.frombuffer(b"".join(msgs), np.uint8),
        "msg_off": msg_off,
        "msg_digest": np.frombuffer(b"".join(m.blake2b_256(x) for x in msgs), np.uint8).reshape(-1, 32),
        "verdict": verdict,
        "key_ok": np.array([m.canonical_point_encoding(v[1]) and not m.blocklisted(v[1]) and m.decode(v[1]) is not None
                            for v in vec], np.uint8),
        "blake_in": np.frombuffer(b"".join(blake_in), np.uint8),
        "blake_off": blake_off,
        "blake_digest": np.frombuffer(b"".join(m.blake2b_256(x) for x in blake_in), np.uint8).reshape(-1, 32),
    }


def main(out=OUT):
    arrays = build()
    np.savez_compressed(out, **arrays)
    print("%s: %d signature vectors (%d accepted), %d BLAKE2b inputs" % (
        out, arrays["verdict"].size, int(arrays["verdict"].sum()), arrays["blake_digest"].shape[0]))


if __name__ == "__main__":
    main(*sys.argv[1:])
