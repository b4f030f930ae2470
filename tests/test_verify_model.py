"""CPU models of the device signature / id checks (py-swirld_b200/csrc/swirld_verify.cuh): the acceptance rules
against libsodium (PyNaCl), the pinned vectors against their generator, and each restructuring the kernel relies on
(32-bit limb field arithmetic, the 16-bit-digit reduction mod L, the doubling-free comb) against plain big integers."""
import os
import random
import sys
import tempfile

import numpy as np
import pytest

import ed25519_model as m

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURE = os.path.join(ROOT, "tests", "golden", "ed25519_vectors.npz")


def _nacl():
    return pytest.importorskip("nacl.bindings")


def _libsodium(sig, msg, pk):
    from nacl.exceptions import CryptoError
    try:
        _nacl().crypto_sign_open(sig + msg, pk)
        return True
    except (CryptoError, ValueError):
        return False


def _vectors():
    z = np.load(FIXTURE)
    for i in range(z["verdict"].size):
        msg = z["msg"][z["msg_off"][i]:z["msg_off"][i + 1]].tobytes()
        yield z, i, z["pk"][i].tobytes(), z["sig"][i].tobytes(), msg


def test_model_matches_libsodium_on_pinned_vectors():
    _nacl()
    seen = set()
    for z, i, pk, sig, msg in _vectors():
        want = bool(z["verdict"][i])
        assert _libsodium(sig, msg, pk) == want, str(z["kind_names"][z["kind"][i]])
        assert m.verify(sig, msg, pk) == want, str(z["kind_names"][z["kind"][i]])
        assert m.blake2b_256(msg) == z["msg_digest"][i].tobytes()
        seen.add((str(z["kind_names"][z["kind"][i]]), want))
    # both verdicts occur where they should
    assert ("valid", True) in seen and ("mixed_order_A_k0mod8", True) in seen
    assert ("mixed_order_A_k_not0mod8", False) in seen and ("identity_R_equation_holds", False) in seen


def test_model_matches_libsodium_on_random_vectors():
    """10 000 random signatures, valid or corrupted (a bit of R, s or msg, another member's key, s + L), through the
    comb model of the kernel's scalar multiplication."""
    b = _nacl()
    rng = random.Random(2024)
    keys = [b.crypto_sign_seed_keypair(rng.randbytes(32)) for _ in range(12)]
    smul = {pk: m.comb_smul_factory(m.decode(pk)) for pk, _ in keys}
    agree = accepted = 0
    for t in range(10000):
        pk, sk = keys[rng.randrange(len(keys))]
        msg = rng.randbytes(rng.randrange(0, 300))
        sig = bytearray(b.crypto_sign(msg, sk)[:64])
        kind = rng.randrange(6)
        if kind == 1:
            sig[rng.randrange(32)] ^= 1 << rng.randrange(8)
        elif kind == 2:
            sig[32 + rng.randrange(32)] ^= 1 << rng.randrange(8)
        elif kind == 3 and msg:
            mm = bytearray(msg); mm[rng.randrange(len(mm))] ^= 1 << rng.randrange(8); msg = bytes(mm)
        elif kind == 4:
            pk = keys[(keys.index((pk, sk)) + 1) % len(keys)][0]
        elif kind == 5 and rng.random() < 0.2:
            s = (int.from_bytes(sig[32:], "little") + m.L) % (1 << 256)
            sig[32:] = s.to_bytes(32, "little")
        sig = bytes(sig)
        want = _libsodium(sig, msg, pk)
        got = m.verify(sig, msg, pk, smul=smul[pk])
        assert got == want, (t, kind)
        agree += 1
        accepted += want
    assert agree == 10000 and 1000 < accepted < 9000


def test_regenerating_the_vectors_gives_the_fixture():
    _nacl()
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import make_verify_vectors as mv
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "v.npz")
        mv.main(out)
        new, old = np.load(out), np.load(FIXTURE)
        assert sorted(new.files) == sorted(old.files)
        for k in old.files:
            assert np.array_equal(new[k], old[k]), k


def test_limb_field_arithmetic_matches_big_integers():
    rng = random.Random(7)
    edge = [0, 1, 2, 18, 19, 37, 38, m.P - 1, m.P, m.P + 1, 2 * m.P, 2 * m.P + 37, 2 ** 255, 2 ** 256 - 39, 2 ** 256 - 38,
            2 ** 256 - 1, 0xFFFFFFFF, 2 ** 224 - 1]
    vals = edge + [rng.getrandbits(256) for _ in range(3000)]
    for i, x in enumerate(vals):
        y = vals[(i * 7 + 3) % len(vals)] if i >= len(edge) else rng.choice(edge)
        a, b = m.to_limbs(x), m.to_limbs(y)
        for op, want in ((m.fe_mul, x * y), (m.fe_add, x + y), (m.fe_sub, x - y)):
            r = op(a, b)
            assert all(0 <= w <= m.MASK32 for w in r)          # stays below 2^256 (not fully reduced)
            assert m.fe_canon(r) == want % m.P
    for x in edge:
        assert m.fe_canon(m.to_limbs(x)) == x % m.P


def test_reduction_mod_L_matches_big_integers():
    rng = random.Random(8)
    hs = [bytes(64), b"\xff" * 64, m.L.to_bytes(64, "little"), (m.L - 1).to_bytes(64, "little"),
          (2 * m.L).to_bytes(64, "little"), (m.L << 256).to_bytes(64, "little")] + [rng.randbytes(64) for _ in range(3000)]
    for h in hs:
        assert m.reduce512(h) == int.from_bytes(h, "little") % m.L


def test_comb_matches_plain_scalar_multiplication():
    """Signed radix-16 recoding and the 64 x 8 table: sum of one mixed addition per digit == [k]P, for the base point,
    an ordinary key and a mixed-order key (a point with a torsion component)."""
    rng = random.Random(9)
    A = m.decode(m.seed_keypair(bytes(32))[0])
    T8 = [t for t in m.small_order_points() if m.encode(m.add(m.add(t, t), m.add(t, t))) != m.encode(m.IDENT)][0]
    for Pt in (m.BASE, m.neg(A), m.add(A, T8)):
        tab = m.comb_table(Pt)
        for k in [0, 1, 7, 8, 9, 15, 16, m.L - 1, 2 ** 253 - 1] + [rng.randrange(m.L) for _ in range(20)]:
            e = m.recode(k)
            assert sum(d << (4 * i) for i, d in enumerate(e)) == k
            assert all(-8 <= d <= 8 for d in e)
            assert m.encode(m.comb_sum(m.IDENT, tab, k)) == m.encode(m.mul(k, Pt))
