"""A small pure-Python Ed25519 written for the tests: libsodium's `crypto_sign_verify_detached` acceptance rules on
plain big integers, signing with an arbitrary scalar (to build mixed-order and small-order vectors), BLAKE2b ids,
and CPU models of the restructurings the verify kernel (py-swirld_b200/csrc/swirld_verify.cuh) relies on:

- field arithmetic on eight 32-bit limbs with values kept below 2^256 (not fully reduced) and 2^256 = 38 (mod p);
- the 512-bit -> mod L reduction, 16 bits at a time with a one-step quotient estimate;
- the comb: a scalar recoded into 64 signed radix-16 digits in [-8, 8], summed from a table of the multiples
  j * 16^i * P (j = 1..8) in affine (y+x, y-x, 2dxy) form by mixed additions only.

Variable-time and slow; for tests only.
"""
from __future__ import annotations

import hashlib

P = 2 ** 255 - 19
L = 2 ** 252 + 27742317777372353535851937790883648493
D = (-121665 * pow(121666, -1, P)) % P
D2 = 2 * D % P
SQRTM1 = pow(2, (P - 1) // 4, P)
MASK32 = 0xFFFFFFFF


# ---------------------------------------------------------------- points (extended coordinates X:Y:Z:T, x = X/Z, y = Y/Z, xy = T/Z)
IDENT = (0, 1, 1, 0)


def add(p, q):
    X1, Y1, Z1, T1 = p
    X2, Y2, Z2, T2 = q
    a = (Y1 - X1) * (Y2 - X2) % P
    b = (Y1 + X1) * (Y2 + X2) % P
    c = T1 * D2 * T2 % P
    d = 2 * Z1 * Z2 % P
    e, f, g, h = b - a, d - c, d + c, b + a
    return (e * f % P, g * h % P, f * g % P, e * h % P)


def neg(p):
    X, Y, Z, T = p
    return (-X % P, Y, Z, -T % P)


def mul(k, p):
    r = IDENT
    while k:
        if k & 1:
            r = add(r, p)
        p = add(p, p)
        k >>= 1
    return r


def affine(p):
    zi = pow(p[2], P - 2, P)
    return p[0] * zi % P, p[1] * zi % P


def encode(p) -> bytes:
    x, y = affine(p)
    return (y | ((x & 1) << 255)).to_bytes(32, "little")


def recover_x(y, sign):
    """libsodium's ge25519_frombytes: x from y (y taken mod p), None when (y^2-1)/(dy^2+1) is not a square.  Like
    libsodium it does not reject x = 0 with the sign bit set."""
    u = (y * y - 1) % P
    v = (D * y * y + 1) % P
    x = u * pow(v, 3, P) * pow(u * pow(v, 7, P), (P - 5) // 8, P) % P
    vxx = v * x * x % P
    if vxx != u:
        if vxx != (-u) % P:
            return None
        x = x * SQRTM1 % P
    if (x & 1) != sign:
        x = (-x) % P
    return x


def decode(s: bytes):
    y = int.from_bytes(s, "little") & ((1 << 255) - 1)
    x = recover_x(y, s[31] >> 7)
    if x is None:
        return None
    y %= P
    return (x, y, 1, x * y % P)


def point_from_y(y, sign=0):
    x = recover_x(y, sign)
    return None if x is None else (x, y % P, 1, x * y % P)


BASE = decode((4 * pow(5, -1, P) % P).to_bytes(32, "little"))


def _small_order_ys():
    """The y of every point of order 1, 2, 4 or 8: [L]Q kills the prime-order part of any point Q."""
    ys, y = {1}, 2
    while len(ys) < 5:
        q = point_from_y(y)
        y += 1
        if q is None:
            continue
        t = mul(L, q)
        for _ in range(3):
            ys.add(affine(t)[1])
            t = add(t, t)
    return sorted(ys)


SMALL_ORDER_YS = _small_order_ys()           # 0 (order 4), 1 (order 1), p - 1 (order 2) and the two of order 8
# libsodium's blocklist: those y, plus the non-canonical p and p + 1; compared with the sign bit masked off
BLOCKLIST_YS = sorted(SMALL_ORDER_YS + [P, P + 1])


def small_order_points():
    """The 8 points of order dividing 8."""
    pts = []
    for y in SMALL_ORDER_YS:
        for sign in (0, 1):
            q = point_from_y(y, sign)
            if q is not None and encode(q) not in [encode(r) for r in pts]:
                pts.append(q)
    return pts


def blocklisted(s: bytes) -> bool:
    return (int.from_bytes(s, "little") & ((1 << 255) - 1)) in BLOCKLIST_YS


def canonical_point_encoding(s: bytes) -> bool:
    return (int.from_bytes(s, "little") & ((1 << 255) - 1)) < P


# ---------------------------------------------------------------- keys, signing, verification (libsodium's rules)
def seed_keypair(seed: bytes):
    """crypto_sign_seed_keypair: (pk, a, prefix)."""
    h = hashlib.sha512(seed).digest()
    a = int.from_bytes(h[:32], "little")
    a &= (1 << 254) - 8
    a |= 1 << 254
    return encode(mul(a, BASE)), a, h[32:]


def challenge(R: bytes, pk: bytes, msg: bytes) -> int:
    return int.from_bytes(hashlib.sha512(R + pk + msg).digest(), "little") % L


def sign_with(a: int, prefix: bytes, pk: bytes, msg: bytes) -> bytes:
    """Ed25519 signing with secret scalar a under the public key bytes pk (which need not be [a]B)."""
    r = int.from_bytes(hashlib.sha512(prefix + msg).digest(), "little") % L
    R = encode(mul(r, BASE))
    s = (r + challenge(R, pk, msg) * a) % L
    return R + s.to_bytes(32, "little")


def verify(sig: bytes, msg: bytes, pk: bytes, smul=None) -> bool:
    """crypto_sign_verify_detached's verdict: s < L; R and A off the small-order blocklist; A canonical and on the
    curve; then the cofactorless check encode([s]B - [k]A) == R byte for byte.  `smul(s, k, A)` may replace the
    plain double scalar multiplication (the comb model)."""
    if len(sig) != 64 or len(pk) != 32:
        return False
    R, s = sig[:32], int.from_bytes(sig[32:], "little")
    if s >= L or not canonical_point_encoding(pk) or blocklisted(pk) or blocklisted(R):
        return False
    A = decode(pk)
    if A is None:
        return False
    k = challenge(R, pk, msg)
    Q = smul(s, k, A) if smul is not None else add(mul(s, BASE), neg(mul(k, A)))
    return encode(Q) == R


def blake2b_256(m: bytes) -> bytes:
    return hashlib.blake2b(m, digest_size=32).digest()


# ---------------------------------------------------------------- the kernel's field arithmetic: 8 x 32-bit limbs, values < 2^256
def to_limbs(x):
    return [(x >> (32 * i)) & MASK32 for i in range(8)]


def from_limbs(v):
    return sum(w << (32 * i) for i, w in enumerate(v))


def fe_add(a, b):
    r, c = [0] * 8, 0
    for i in range(8):
        c += a[i] + b[i]
        r[i], c = c & MASK32, c >> 32
    c *= 38                                   # 2^256 = 38 (mod p)
    for i in range(8):
        c += r[i]
        r[i], c = c & MASK32, c >> 32
    r[0] += 38 * c                            # a second carry leaves r < 38: no further carry
    assert r[0] <= MASK32
    return r


def fe_sub(a, b):
    r, br = [0] * 8, 0
    for i in range(8):
        t = a[i] - b[i] - br
        r[i], br = t & MASK32, 1 if t < 0 else 0
    if br:                                    # r = a - b + 2^256: take 38 away
        for rep in range(2):                  # a second borrow (r < 38) wraps again: 38 more
            br = 38
            for i in range(8):
                t = r[i] - br
                r[i], br = t & MASK32, 1 if t < 0 else 0
            if not br:
                break
    return r


def fe_mul(a, b):
    t = [0] * 16
    for i in range(8):
        c = 0
        for j in range(8):
            c = a[i] * b[j] + t[i + j] + (c >> 32)
            assert c < 1 << 64
            t[i + j] = c & MASK32
        t[i + 8] = c >> 32
    r, c = [0] * 8, 0
    for i in range(8):
        c = t[i + 8] * 38 + t[i] + (c >> 32)
        r[i] = c & MASK32
    c = (c >> 32) * 38
    for i in range(8):
        c += r[i]
        r[i], c = c & MASK32, c >> 32
    r[0] += 38 * c
    assert r[0] <= MASK32
    return r


def fe_canon(a):
    x = from_limbs(a)
    for _ in range(2):                        # x < 2^256 = 2p + 38
        if x >= P:
            x -= P
    return x


# ---------------------------------------------------------------- the kernel's k = SHA-512(...) mod L: 16 bits at a time
def reduce512(h: bytes) -> int:
    """Horner over the 32 16-bit digits, most significant first: t = r * 2^16 + digit < 2^269, q = t >> 252 over-
    estimates t // L by at most one (L > 2^252, and t * (L - 2^252) / 2^504 < 1), so t - q L is in [-L, L)."""
    x = int.from_bytes(h, "little")
    r = 0
    for i in range(31, -1, -1):
        t = (r << 16) | ((x >> (16 * i)) & 0xFFFF)
        q = t >> 252
        r = t - q * L
        if r < 0:
            r += L
        assert 0 <= r < L
    return r


# ---------------------------------------------------------------- the comb
def recode(k: int):
    """64 signed radix-16 digits e with sum(e[i] 16^i) = k; e[i] in [-8, 7] for i < 63, e[63] in [-8, 8] (k < 2^255)."""
    e = [(k >> (4 * i)) & 15 for i in range(64)]
    carry = 0
    for i in range(63):
        e[i] += carry
        carry = (e[i] + 8) >> 4
        e[i] -= carry << 4
    e[63] += carry
    return e


def comb_table(Pt):
    """tab[i][j - 1] = j * 16^i * Pt in affine (y+x, y-x, 2dxy) form, i = 0..63, j = 1..8."""
    tab, Q = [], Pt
    for i in range(64):
        row, M = [], Q
        for j in range(1, 9):
            x, y = affine(M)
            row.append(((y + x) % P, (y - x) % P, D2 * x * y % P))
            M = add(M, Q)
        tab.append(row)
        for _ in range(4):
            Q = add(Q, Q)
    return tab


def madd(p, q, negate):
    """Extended + affine (y+x, y-x, 2dxy); negate: add -q instead (swap y+x / y-x, negate 2dxy)."""
    X1, Y1, Z1, T1 = p
    ypx, ymx, xy2d = q
    if negate:
        ypx, ymx = ymx, ypx
    a = (Y1 - X1) * ymx % P
    b = (Y1 + X1) * ypx % P
    c = T1 * xy2d % P
    d = 2 * Z1 % P
    if negate:
        c = -c
    e, f, g, h = b - a, d - c, d + c, b + a
    return (e * f % P, g * h % P, f * g % P, e * h % P)


def comb_sum(acc, tab, k):
    for i, e in enumerate(recode(k)):
        if e:
            acc = madd(acc, tab[i][abs(e) - 1], e < 0)
    return acc


_BASE_TAB = None


def comb_smul_factory(A):
    """smul(s, k, A) for verify(): [s]B + [k](-A) from the two comb tables (B's shared, -A's per member)."""
    global _BASE_TAB
    if _BASE_TAB is None:
        _BASE_TAB = comb_table(BASE)
    tab_negA = comb_table(neg(A))
    return lambda s, k, _A: comb_sum(comb_sum(IDENT, _BASE_TAB, s), tab_negA, k)
