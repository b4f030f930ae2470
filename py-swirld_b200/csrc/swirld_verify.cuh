// swirld_verify.cuh -- is_valid_event's two crypto checks (swirld.py:97-103) for a batch of events, one thread per
// event: the Ed25519 signature with the verdict of libsodium's crypto_sign_verify_detached, and id == BLAKE2b-256 of
// the pickled event.  Integer-only; 64-bit hash words are pairs of 32-bit registers (funnel shifts for the rotates),
// field elements are eight 32-bit limbs multiplied with 32 x 32 -> 64-bit multiply-adds.
//
// Acceptance rules (libsodium's, which differ from other Ed25519 implementations at the edges):
//   s < L;  R and A not on the small-order blocklist (sign bit ignored);  A canonical (y < p) and on the curve;
//   k = SHA-512(R || A || msg) mod L;  accept iff encode([s]B - [k]A) == R byte for byte (cofactorless; the byte
//   comparison is what rejects a non-canonical or off-curve R).
// Scalar multiplication is a comb without doublings: [s]B and [k](-A) are sums of one table entry per radix-16 signed
// digit, j * 16^i * P for j = 1..8 in affine (y+x, y-x, 2dxy) form -- 128 mixed additions per event.  The table of B
// lives in shared memory (48 KB per CTA); the table of -A of every member is built once by sw_set_member_keys
// (48 KB per member in device memory).  Public data only: the code is variable-time, like libsodium's verify.
// The math is __host__ __device__ so that it can be checked on the CPU as well.
#pragma once
#include <cstdint>
#include <cstring>

#define SWV_HD __host__ __device__ __forceinline__

namespace swv {

typedef uint32_t u32;
typedef uint64_t u64;

// ---------------------------------------------------------------- field: Z / (2^255 - 19), values < 2^256
struct fe { u32 v[8]; };

struct __align__(16) Precomp { fe ypx, ymx, xy2d; };            // affine (y + x, y - x, 2 d x y)
struct Point { fe X, Y, Z, T; };                                 // extended: x = X/Z, y = Y/Z, x y = T/Z

constexpr int COMB_ENTRIES = 64 * 8;                             // per table: 64 radix-16 positions x multiples 1..8

__host__ __device__ inline const u32 *c_d2() {
    static constexpr u32 v[8] = {0x26b2f159u, 0xebd69b94u, 0x8283b156u, 0x00e0149au, 0xeef3d130u, 0x198e80f2u, 0x56dffce7u, 0x2406d9dcu};
    return v;
}

SWV_HD void fe_set(fe &r, const u32 *c) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = c[i];
}
SWV_HD void fe_one(fe &r) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = i == 0;
}
SWV_HD void fe_zero(fe &r) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = 0;
}

SWV_HD void fe_add(fe &r, const fe &a, const fe &b) {
    u64 c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { c += (u64)a.v[i] + b.v[i]; r.v[i] = (u32)c; c >>= 32; }
    c *= 38;                                                      // 2^256 = 38 (mod p)
#pragma unroll
    for (int i = 0; i < 8; i++) { c += r.v[i]; r.v[i] = (u32)c; c >>= 32; }
    r.v[0] += (u32)c * 38;                                        // a second carry leaves r < 38
}

SWV_HD void fe_sub(fe &r, const fe &a, const fe &b) {
    u64 t = 0;
    u32 br = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { t = (u64)a.v[i] - b.v[i] - br; r.v[i] = (u32)t; br = (u32)(t >> 63); }
    if (br) {                                                     // r = a - b + 2^256: take 38 away (twice if that wraps)
        br = 38;
#pragma unroll
        for (int i = 0; i < 8; i++) { t = (u64)r.v[i] - br; r.v[i] = (u32)t; br = (u32)(t >> 63); }
        r.v[0] -= br * 38;                                        // (after a wrap r >= 2^256 - 38: no borrow)
    }
}

SWV_HD void fe_mul(fe &r, const fe &a, const fe &b) {
    u32 t[16];
#pragma unroll
    for (int i = 0; i < 16; i++) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        u64 c = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            c = (u64)a.v[i] * b.v[j] + t[i + j] + (c >> 32);       // <= (2^32-1)^2 + 2 (2^32-1) = 2^64 - 1
            t[i + j] = (u32)c;
        }
        t[i + 8] = (u32)(c >> 32);
    }
    u64 c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { c = (u64)t[i + 8] * 38 + t[i] + (c >> 32); r.v[i] = (u32)c; }
    c = (c >> 32) * 38;
#pragma unroll
    for (int i = 0; i < 8; i++) { c += r.v[i]; r.v[i] = (u32)c; c >>= 32; }
    r.v[0] += (u32)c * 38;
}

SWV_HD void fe_sq(fe &r, const fe &a) { fe_mul(r, a, a); }

SWV_HD void fe_sqn(fe &r, const fe &a, int n) {
    fe_sq(r, a);
    for (int i = 1; i < n; i++) fe_sq(r, r);
}

// z^(2^250 - 1) and z^11: the common part of the inversion and square-root chains
SWV_HD void fe_pow_250(fe &z250, fe &z11, const fe &z) {
    fe z2, t, z9, z5, z10, z20, z40, z50, z100, z200;
    fe_sq(z2, z);
    fe_sqn(t, z2, 2);
    fe_mul(z9, t, z);
    fe_mul(z11, z9, z2);
    fe_sq(t, z11);
    fe_mul(z5, t, z9);                                            // 2^5 - 1
    fe_sqn(t, z5, 5);   fe_mul(z10, t, z5);
    fe_sqn(t, z10, 10); fe_mul(z20, t, z10);
    fe_sqn(t, z20, 20); fe_mul(z40, t, z20);
    fe_sqn(t, z40, 10); fe_mul(z50, t, z10);
    fe_sqn(t, z50, 50); fe_mul(z100, t, z50);
    fe_sqn(t, z100, 100); fe_mul(z200, t, z100);
    fe_sqn(t, z200, 50); fe_mul(z250, t, z50);
}

SWV_HD void fe_inv(fe &r, const fe &z) {                          // z^(p - 2) = z^(2^255 - 21)
    fe z250, z11, t;
    fe_pow_250(z250, z11, z);
    fe_sqn(t, z250, 5);
    fe_mul(r, t, z11);
}

SWV_HD void fe_pow2523(fe &r, const fe &z) {                      // z^((p - 5) / 8) = z^(2^252 - 3)
    fe z250, z11, t;
    fe_pow_250(z250, z11, z);
    fe_sqn(t, z250, 2);
    fe_mul(r, t, z);
}

// fully reduced: [0, p)  (a < 2^256 = 2p + 38: at most two subtractions)
SWV_HD void fe_canon(fe &r, const fe &a) {
    r = a;
    for (int rep = 0; rep < 2; rep++) {
        fe s;
        u64 t;
        u32 br = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const u32 pi = i == 0 ? 0xffffffedu : i == 7 ? 0x7fffffffu : 0xffffffffu;
            t = (u64)r.v[i] - pi - br; s.v[i] = (u32)t; br = (u32)(t >> 63);
        }
        if (br) break;
        r = s;
    }
}

SWV_HD bool fe_iszero(const fe &a) {
    fe c;
    fe_canon(c, a);
    u32 o = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) o |= c.v[i];
    return o == 0;
}

SWV_HD void fe_neg(fe &r, const fe &a) { fe z; fe_zero(z); fe_sub(r, z, a); }

// ---------------------------------------------------------------- points
SWV_HD void pt_identity(Point &p) { fe_zero(p.X); fe_one(p.Y); fe_one(p.Z); fe_zero(p.T); }

// p + q with q affine (y+x, y-x, 2dxy); negate: p - q.  7 multiplications; complete on the curve.
SWV_HD void pt_madd(Point &r, const Point &p, const Precomp &q, bool negate) {
    fe a, b, c, d, e, f, g, h;
    fe_sub(a, p.Y, p.X);
    fe_add(b, p.Y, p.X);
    fe_mul(a, a, negate ? q.ypx : q.ymx);
    fe_mul(b, b, negate ? q.ymx : q.ypx);
    fe_mul(c, p.T, q.xy2d);
    fe_add(d, p.Z, p.Z);
    fe_sub(e, b, a);
    fe_add(h, b, a);
    fe_sub(f, d, c);
    fe_add(g, d, c);
    if (negate) { fe x = f; f = g; g = x; }
    fe_mul(r.X, e, f);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    fe_mul(r.T, e, h);
}

SWV_HD void pt_dbl(Point &r, const Point &p) {
    fe xx, yy, zz2, s, ss, e, f, g, h;
    fe_sq(xx, p.X);
    fe_sq(yy, p.Y);
    fe_sq(zz2, p.Z);
    fe_add(zz2, zz2, zz2);
    fe_add(s, p.X, p.Y);
    fe_sq(ss, s);
    fe_add(h, yy, xx);                                            // Y^2 + X^2
    fe_sub(g, yy, xx);                                            // Y^2 - X^2
    fe_sub(e, ss, h);                                             // 2 X Y
    fe_sub(f, zz2, g);                                            // 2 Z^2 - (Y^2 - X^2)
    fe_mul(r.X, e, f);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    fe_mul(r.T, e, h);
}

SWV_HD void pt_to_precomp(Precomp &q, const Point &p) {
    fe zi, x, y;
    fe_inv(zi, p.Z);
    fe_mul(x, p.X, zi);
    fe_mul(y, p.Y, zi);
    fe_add(q.ypx, y, x);
    fe_sub(q.ymx, y, x);
    fe d2;
    fe_set(d2, c_d2());
    fe_mul(q.xy2d, x, y);
    fe_mul(q.xy2d, q.xy2d, d2);
}

SWV_HD u32 load_le32(const uint8_t *p) { return (u32)p[0] | (u32)p[1] << 8 | (u32)p[2] << 16 | (u32)p[3] << 24; }

// libsodium's ge25519_has_small_order: the encoding's y (sign bit ignored) is one of 7 values
SWV_HD bool blocklisted(const u32 *s) {
    static constexpr u32 BL[7][8] = {
        {0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u},
        {0x00000001u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u},
        {0x8f95e826u, 0xb027b2c2u, 0x89f4c345u, 0xf098eff2u, 0x05acdfd5u, 0x3933c6d3u, 0x880238b1u, 0x05fc536du},
        {0x706a17c7u, 0x4fd84d3du, 0x760b3cbau, 0x0f67100du, 0xfa53202au, 0xc6cc392cu, 0x77fdc74eu, 0x7a03ac92u},
        {0xffffffecu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0x7fffffffu},  // p - 1
        {0xffffffedu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0x7fffffffu},  // p
        {0xffffffeeu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0x7fffffffu},  // p + 1
    };
    for (int j = 0; j < 7; j++) {
        u32 o = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) o |= (i == 7 ? s[i] & 0x7fffffffu : s[i]) ^ BL[j][i];
        if (o == 0) return true;
    }
    return false;
}

// y of an encoding (sign bit masked) < p
SWV_HD bool canonical_y(const u32 *s) {
    if ((s[7] & 0x7fffffffu) != 0x7fffffffu) return true;
    for (int i = 1; i < 7; i++) if (s[i] != 0xffffffffu) return true;
    return s[0] < 0xffffffedu;
}

// libsodium's ge25519_frombytes (y taken mod p, x = 0 with the sign bit set not rejected); negate: the point's negative
SWV_HD bool pt_decode(Point &r, const u32 *s, bool negate) {
    fe y, u, v, v3, x, t, one, d2, d;
    fe_set(y, s);
    y.v[7] &= 0x7fffffffu;
    fe_one(one);
    fe_set(d2, c_d2());
    const fe dh = {{0x135978a3u, 0x75eb4dcau, 0x4141d8abu, 0x00700a4du, 0x7779e898u, 0x8cc74079u, 0x2b6ffe73u, 0x52036ceeu}};
    d = dh;
    fe_sq(u, y);
    fe_mul(v, u, d);
    fe_sub(u, u, one);                                            // u = y^2 - 1
    fe_add(v, v, one);                                            // v = d y^2 + 1
    fe_sq(v3, v);
    fe_mul(v3, v3, v);                                            // v^3
    fe_sq(x, v3);
    fe_mul(x, x, v);
    fe_mul(x, x, u);                                              // u v^7
    fe_pow2523(x, x);
    fe_mul(x, x, v3);
    fe_mul(x, x, u);                                              // u v^3 (u v^7)^((p-5)/8)
    fe_sq(t, x);
    fe_mul(t, t, v);                                              // v x^2
    fe chk;
    fe_sub(chk, t, u);
    if (!fe_iszero(chk)) {
        fe_add(chk, t, u);
        if (!fe_iszero(chk)) return false;
        const fe sm1 = {{0x4a0ea0b0u, 0xc4ee1b27u, 0xad2fe478u, 0x2f431806u, 0x3dfbd7a7u, 0x2b4d0099u, 0x4fc1df0bu, 0x2b832480u}};
        fe_mul(x, x, sm1);
    }
    fe xc;
    fe_canon(xc, x);
    const u32 want = (s[7] >> 31) ^ (negate ? 1u : 0u);           // parity of the x we keep
    if ((xc.v[0] & 1u) != want) fe_neg(x, xc); else x = xc;
    r.X = x;
    r.Y = y;
    fe_one(r.Z);
    fe_mul(r.T, x, y);
    return true;
}

// encode(p) == the 32 bytes s (as LE words): y canonical and equal, x's parity equal to the sign bit
SWV_HD bool pt_encodes_to(const Point &p, const u32 *s) {
    fe zi, x, y;
    fe_inv(zi, p.Z);
    fe_mul(x, p.X, zi);
    fe_mul(y, p.Y, zi);
    fe_canon(x, x);
    fe_canon(y, y);
    u32 o = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) o |= y.v[i] ^ (i == 7 ? s[i] & 0x7fffffffu : s[i]);
    return o == 0 && (x.v[0] & 1u) == (s[7] >> 31);
}

// ---------------------------------------------------------------- scalars mod L = 2^252 + 27742317777372353535851937790883648493
__host__ __device__ inline const u32 *c_L() {
    static constexpr u32 v[8] = {0x5cf5d3edu, 0x5812631au, 0xa2f79cd6u, 0x14def9deu, 0u, 0u, 0u, 0x10000000u};
    return v;
}

SWV_HD bool sc_lt_L(const u32 *s) {
    const u32 *Lw = c_L();
    for (int i = 7; i >= 0; i--) {
        if (s[i] < Lw[i]) return true;
        if (s[i] > Lw[i]) return false;
    }
    return false;
}

// k = h mod L for the 64-byte little-endian h: Horner over 16-bit digits, most significant first.  t = r 2^16 + digit
// < 2^269; q = t >> 252 over-estimates t / L by at most one, so t - q L is in [-L, L): add L back when negative.
SWV_HD void sc_reduce512(u32 *k, const u32 *h16w) {
    const u32 *Lw = c_L();
    u32 r[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int d = 31; d >= 0; d--) {
        const u32 digit = (h16w[d >> 1] >> (16 * (d & 1))) & 0xffffu;
        // t = r << 16 | digit (9 limbs: r < 2^253)
        u32 t[9];
        t[0] = (r[0] << 16) | digit;
#pragma unroll
        for (int i = 1; i < 9; i++) t[i] = (r[i] << 16) | (r[i - 1] >> 16);
        const u32 q = (t[8] << 4) | (t[7] >> 28);
        // t -= q L
        u64 c = 0;
        u32 br = 0;
#pragma unroll
        for (int i = 0; i < 9; i++) {
            c = (u64)q * (i < 8 ? Lw[i] : 0u) + (c >> 32);
            const u64 s = (u64)t[i] - (u32)c - br;
            r[i] = (u32)s;
            br = (u32)(s >> 63);
        }
        if (br) {                                                 // negative: + L
            u64 a = 0;
#pragma unroll
            for (int i = 0; i < 9; i++) { a += (u64)r[i] + (i < 8 ? Lw[i] : 0u); r[i] = (u32)a; a >>= 32; }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) k[i] = r[i];
}

// ---------------------------------------------------------------- 64-bit words as 32-bit pairs
struct w64 { u32 lo, hi; };

SWV_HD w64 mk64(u64 x) { return w64{(u32)x, (u32)(x >> 32)}; }
SWV_HD w64 add64(w64 a, w64 b) {
    const u32 lo = a.lo + b.lo;
    return w64{lo, a.hi + b.hi + (lo < a.lo)};
}
SWV_HD w64 xor64(w64 a, w64 b) { return w64{a.lo ^ b.lo, a.hi ^ b.hi}; }
SWV_HD w64 and64(w64 a, w64 b) { return w64{a.lo & b.lo, a.hi & b.hi}; }
SWV_HD w64 not64(w64 a) { return w64{~a.lo, ~a.hi}; }
SWV_HD u32 fshr(u32 lo, u32 hi, int n) {                          // (hi:lo) >> n, low word; 0 < n < 32
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, n);
#else
    return (lo >> n) | (hi << (32 - n));
#endif
}
SWV_HD w64 rotr64(w64 a, int n) {                                 // n compile-time after inlining
    if (n == 32) return w64{a.hi, a.lo};
    if (n < 32) return w64{fshr(a.lo, a.hi, n), fshr(a.hi, a.lo, n)};
    return w64{fshr(a.hi, a.lo, n - 32), fshr(a.lo, a.hi, n - 32)};
}
SWV_HD w64 shr64(w64 a, int n) {                                  // 0 < n < 32
    return w64{fshr(a.lo, a.hi, n), a.hi >> n};
}

// ---------------------------------------------------------------- SHA-512 of R || A || msg
__host__ __device__ inline u64 sha512_k(int i) {
    static constexpr u64 K[80] = {
        0x428a2f98d728ae22ull, 0x7137449123ef65cdull, 0xb5c0fbcfec4d3b2full, 0xe9b5dba58189dbbcull, 0x3956c25bf348b538ull, 0x59f111f1b605d019ull, 0x923f82a4af194f9bull, 0xab1c5ed5da6d8118ull,
        0xd807aa98a3030242ull, 0x12835b0145706fbeull, 0x243185be4ee4b28cull, 0x550c7dc3d5ffb4e2ull, 0x72be5d74f27b896full, 0x80deb1fe3b1696b1ull, 0x9bdc06a725c71235ull, 0xc19bf174cf692694ull,
        0xe49b69c19ef14ad2ull, 0xefbe4786384f25e3ull, 0x0fc19dc68b8cd5b5ull, 0x240ca1cc77ac9c65ull, 0x2de92c6f592b0275ull, 0x4a7484aa6ea6e483ull, 0x5cb0a9dcbd41fbd4ull, 0x76f988da831153b5ull,
        0x983e5152ee66dfabull, 0xa831c66d2db43210ull, 0xb00327c898fb213full, 0xbf597fc7beef0ee4ull, 0xc6e00bf33da88fc2ull, 0xd5a79147930aa725ull, 0x06ca6351e003826full, 0x142929670a0e6e70ull,
        0x27b70a8546d22ffcull, 0x2e1b21385c26c926ull, 0x4d2c6dfc5ac42aedull, 0x53380d139d95b3dfull, 0x650a73548baf63deull, 0x766a0abb3c77b2a8ull, 0x81c2c92e47edaee6ull, 0x92722c851482353bull,
        0xa2bfe8a14cf10364ull, 0xa81a664bbc423001ull, 0xc24b8b70d0f89791ull, 0xc76c51a30654be30ull, 0xd192e819d6ef5218ull, 0xd69906245565a910ull, 0xf40e35855771202aull, 0x106aa07032bbd1b8ull,
        0x19a4c116b8d2d0c8ull, 0x1e376c085141ab53ull, 0x2748774cdf8eeb99ull, 0x34b0bcb5e19b48a8ull, 0x391c0cb3c5c95a63ull, 0x4ed8aa4ae3418acbull, 0x5b9cca4f7763e373ull, 0x682e6ff3d6b2b8a3ull,
        0x748f82ee5defb2fcull, 0x78a5636f43172f60ull, 0x84c87814a1f0ab72ull, 0x8cc702081a6439ecull, 0x90befffa23631e28ull, 0xa4506cebde82bde9ull, 0xbef9a3f7b2c67915ull, 0xc67178f2e372532bull,
        0xca273eceea26619cull, 0xd186b8c721c0c207ull, 0xeada7dd6cde0eb1eull, 0xf57d4f7fee6ed178ull, 0x06f067aa72176fbaull, 0x0a637dc5a2c898a6ull, 0x113f9804bef90daeull, 0x1b710b35131c471bull,
        0x28db77f523047d84ull, 0x32caab7b40c72493ull, 0x3c9ebe0a15c9bebcull, 0x431d67c49c100d4cull, 0x4cc5d4becb3e42b6ull, 0x597f299cfc657e2aull, 0x5fcb6fab3ad6faecull, 0x6c44198c4a475817ull};
    return K[i];
}
__host__ __device__ inline u64 iv512(int i) {                     // SHA-512's initial value, also BLAKE2b's IV
    static constexpr u64 IV[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                                  0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
    return IV[i];
}

SWV_HD void sha512_block(w64 *h, w64 *w) {                        // w[16]: the block, big-endian words (clobbered)
    w64 a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
    for (int i = 0; i < 80; i++) {
        w64 wi;
        if (i < 16) wi = w[i];
        else {
            const w64 w15 = w[(i - 15) & 15], w2 = w[(i - 2) & 15];
            const w64 s0 = xor64(xor64(rotr64(w15, 1), rotr64(w15, 8)), shr64(w15, 7));
            const w64 s1 = xor64(xor64(rotr64(w2, 19), rotr64(w2, 61)), shr64(w2, 6));
            wi = add64(add64(w[i & 15], s0), add64(w[(i - 7) & 15], s1));
            w[i & 15] = wi;
        }
        const w64 S1 = xor64(xor64(rotr64(e, 14), rotr64(e, 18)), rotr64(e, 41));
        const w64 ch = xor64(and64(e, f), and64(not64(e), g));
        const w64 t1 = add64(add64(add64(hh, S1), add64(ch, mk64(sha512_k(i)))), wi);
        const w64 S0 = xor64(xor64(rotr64(a, 28), rotr64(a, 34)), rotr64(a, 39));
        const w64 mj = xor64(xor64(and64(a, b), and64(a, c)), and64(b, c));
        const w64 t2 = add64(S0, mj);
        hh = g; g = f; f = e; e = add64(d, t1); d = c; c = b; b = a; a = add64(t1, t2);
    }
    h[0] = add64(h[0], a); h[1] = add64(h[1], b); h[2] = add64(h[2], c); h[3] = add64(h[3], d);
    h[4] = add64(h[4], e); h[5] = add64(h[5], f); h[6] = add64(h[6], g); h[7] = add64(h[7], hh);
}

SWV_HD u32 bswap32(u32 x) {
#ifdef __CUDA_ARCH__
    return __byte_perm(x, 0, 0x0123);
#else
    return __builtin_bswap32(x);
#endif
}

// SHA-512(R || A || msg) as 16 little-endian 32-bit words (the byte order of the 512-bit integer k is read from)
SWV_HD void sha512_ram(u32 *out16, const uint8_t *R, const uint8_t *A, const uint8_t *msg, u64 mlen) {
    w64 h[8];
    for (int i = 0; i < 8; i++) h[i] = mk64(iv512(i));
    const u64 len = 64 + mlen;
    const u64 nb = (len + 17 + 127) / 128;
    for (u64 b = 0; b < nb; b++) {
        w64 w[16];
        for (int j = 0; j < 16; j++) {
            u32 hw = 0, lw = 0;
            for (int k = 0; k < 8; k++) {
                const u64 pos = b * 128 + j * 8 + k;
                u32 byte;
                if (pos < 32) byte = R[pos];
                else if (pos < 64) byte = A[pos - 32];
                else if (pos < len) byte = msg[pos - 64];
                else byte = pos == len ? 0x80u : 0u;
                if (k < 4) hw = hw << 8 | byte; else lw = lw << 8 | byte;
            }
            w[j] = w64{lw, hw};
        }
        if (b == nb - 1) w[15] = mk64(len << 3), w[14] = mk64(len >> 61);
        sha512_block(h, w);
    }
    for (int i = 0; i < 8; i++) {                                 // digest bytes = big-endian words
        const u32 hi = h[i].hi, lo = h[i].lo;
        out16[2 * i] = bswap32(hi);
        out16[2 * i + 1] = bswap32(lo);
    }
}

// ---------------------------------------------------------------- BLAKE2b-256, unkeyed (crypto_generichash, swirld.py:95)
SWV_HD void b2_g(w64 *v, int a, int b, int c, int d, w64 x, w64 y) {
    v[a] = add64(add64(v[a], v[b]), x); v[d] = rotr64(xor64(v[d], v[a]), 32);
    v[c] = add64(v[c], v[d]);           v[b] = rotr64(xor64(v[b], v[c]), 24);
    v[a] = add64(add64(v[a], v[b]), y); v[d] = rotr64(xor64(v[d], v[a]), 16);
    v[c] = add64(v[c], v[d]);           v[b] = rotr64(xor64(v[b], v[c]), 63);
}

__host__ __device__ inline int b2_sigma(int r, int i) {
    static constexpr uint8_t S[10][16] = {
        {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3},
        {11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4}, {7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8},
        {9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13}, {2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9},
        {12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11}, {13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10},
        {6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5}, {10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0}};
    return S[r % 10][i];
}

// digest bytes 0..31 as 8 little-endian words
SWV_HD void blake2b_256(u32 *out8, const uint8_t *m, u64 n) {
    w64 h[8];
    for (int i = 0; i < 8; i++) h[i] = mk64(iv512(i));
    h[0] = xor64(h[0], mk64(0x01010020ull));                     // depth 1, fanout 1, no key, 32-byte digest
    const u64 nb = n == 0 ? 1 : (n + 127) / 128;
    for (u64 b = 0; b < nb; b++) {
        w64 mw[16];
        for (int j = 0; j < 16; j++) {
            u32 lw = 0, hw = 0;
            for (int k = 7; k >= 0; k--) {
                const u64 pos = b * 128 + j * 8 + k;
                const u32 byte = pos < n ? m[pos] : 0u;
                if (k >= 4) hw = hw << 8 | byte; else lw = lw << 8 | byte;
            }
            mw[j] = w64{lw, hw};
        }
        const bool last = b == nb - 1;
        const u64 t = last ? n : (b + 1) * 128;
        w64 v[16];
        for (int i = 0; i < 8; i++) { v[i] = h[i]; v[i + 8] = mk64(iv512(i)); }
        v[12] = xor64(v[12], mk64(t));
        if (last) v[14] = not64(v[14]);
        for (int r = 0; r < 12; r++) {
            b2_g(v, 0, 4, 8, 12, mw[b2_sigma(r, 0)], mw[b2_sigma(r, 1)]);
            b2_g(v, 1, 5, 9, 13, mw[b2_sigma(r, 2)], mw[b2_sigma(r, 3)]);
            b2_g(v, 2, 6, 10, 14, mw[b2_sigma(r, 4)], mw[b2_sigma(r, 5)]);
            b2_g(v, 3, 7, 11, 15, mw[b2_sigma(r, 6)], mw[b2_sigma(r, 7)]);
            b2_g(v, 0, 5, 10, 15, mw[b2_sigma(r, 8)], mw[b2_sigma(r, 9)]);
            b2_g(v, 1, 6, 11, 12, mw[b2_sigma(r, 10)], mw[b2_sigma(r, 11)]);
            b2_g(v, 2, 7, 8, 13, mw[b2_sigma(r, 12)], mw[b2_sigma(r, 13)]);
            b2_g(v, 3, 4, 9, 14, mw[b2_sigma(r, 14)], mw[b2_sigma(r, 15)]);
        }
        for (int i = 0; i < 8; i++) h[i] = xor64(h[i], xor64(v[i], v[i + 8]));
    }
    for (int i = 0; i < 4; i++) { out8[2 * i] = h[i].lo; out8[2 * i + 1] = h[i].hi; }
}

// ---------------------------------------------------------------- the comb: [s]B + [k](-A), 128 mixed additions
// Digits are recoded on the fly: the scalar is shifted right 4 bits per position, digit in [-8, 8] (the carry goes
// into the next position).  tabB / tabA: COMB_ENTRIES entries, [i * 8 + j - 1] = j 16^i P.
template <typename TB, typename TA>
SWV_HD void comb_double_scalar(Point &acc, u32 *s, u32 *k, const TB &tabB, const TA &tabA) {
    pt_identity(acc);
    int cs = 0, ck = 0;
    for (int i = 0; i < 64; i++) {
        int ds = (int)(s[0] & 15u) + cs, dk = (int)(k[0] & 15u) + ck;
#pragma unroll
        for (int w = 0; w < 7; w++) { s[w] = (s[w] >> 4) | (s[w + 1] << 28); k[w] = (k[w] >> 4) | (k[w + 1] << 28); }
        s[7] >>= 4;
        k[7] >>= 4;
        if (i < 63) {
            cs = (ds + 8) >> 4; ds -= cs << 4;
            ck = (dk + 8) >> 4; dk -= ck << 4;
        }
        if (ds) { const Precomp q = tabB(i * 8 + (ds < 0 ? -ds : ds) - 1); pt_madd(acc, acc, q, ds < 0); }
        if (dk) { const Precomp q = tabA(i * 8 + (dk < 0 ? -dk : dk) - 1); pt_madd(acc, acc, q, dk < 0); }
    }
}

// The signature check of one event, A's table given (the member's key passed the key checks).
template <typename TB, typename TA>
SWV_HD bool ed25519_verify(const uint8_t *sig, const uint8_t *pk, const uint8_t *msg, u64 mlen, const TB &tabB, const TA &tabA) {
    u32 Rw[8], s[8], h[16], k[8];
    for (int i = 0; i < 8; i++) { Rw[i] = load_le32(sig + 4 * i); s[i] = load_le32(sig + 32 + 4 * i); }
    if (!sc_lt_L(s) || blocklisted(Rw)) return false;
    sha512_ram(h, sig, pk, msg, mlen);
    sc_reduce512(k, h);
    Point acc;
    comb_double_scalar(acc, s, k, tabB, tabA);
    return pt_encodes_to(acc, Rw);
}

// A member key: canonical, off the blocklist, on the curve.  Writes -A (B for the base point) in affine form.
SWV_HD bool key_decode(Point &negA, const uint8_t *pk, bool is_base) {
    u32 w[8];
    for (int i = 0; i < 8; i++) w[i] = load_le32(pk + 4 * i);
    if (!is_base && (!canonical_y(w) || blocklisted(w))) return false;
    return pt_decode(negA, w, !is_base);
}

// One 8-entry row of a comb table: j * 16^i * P, j = 1..8 (P affine: Z = 1)
SWV_HD void comb_row(Precomp *out8, const Point &P, int i) {
    Point Q = P;
    for (int t = 0; t < 4 * i; t++) pt_dbl(Q, Q);
    Precomp q1;
    pt_to_precomp(q1, Q);
    out8[0] = q1;
    Point M = Q;
    for (int j = 2; j <= 8; j++) {
        pt_madd(M, M, q1, false);
        pt_to_precomp(out8[j - 1], M);
    }
}

}  // namespace swv

// ---------------------------------------------------------------- kernels
struct SwVerifyArgs {
    int n, M;
    const int32_t *sel;          // thread j checks event sel[j] (NULL: event j)
    const int32_t *creator;
    const uint8_t *sig, *msg, *ids, *wire;
    const int64_t *msg_off, *wire_off;
    const uint8_t *pk, *keyok;   // M x 32, M
    const swv::Precomp *tab;     // (M + 1) x COMB_ENTRIES: members' -A, then B
    uint8_t *status;             // indexed like the input events
};

// keys: thread r < M decodes member r's key, r == M the base point; writes the affine point and the verdict
__global__ void k_verify_keys(const uint8_t *pk, int M, swv::Point *base, uint8_t *keyok) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > M) return;
    uint8_t enc[32];                                              // B: y = 4/5, x even: 58 66 66 .. 66
    for (int i = 0; i < 32; i++) enc[i] = r < M ? pk[(size_t)32 * r + i] : i == 0 ? 0x58 : 0x66;
    swv::Point P;
    const bool ok = swv::key_decode(P, enc, r == M);
    if (ok) base[r] = P;
    keyok[r] = ok ? 1 : 0;
}

// tables: one thread per (row r <= M, radix-16 position i)
__global__ void k_verify_table(const swv::Point *base, const uint8_t *keyok, int M, swv::Precomp *tab) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (M + 1) * 64) return;
    const int r = g >> 6, i = g & 63;
    if (!keyok[r]) return;
    swv::comb_row(tab + (size_t)r * swv::COMB_ENTRIES + i * 8, base[r], i);
}

constexpr int SWV_THREADS = 128;

__global__ void __launch_bounds__(SWV_THREADS) k_verify(SwVerifyArgs a) {
    extern __shared__ uint4 swv_smem[];
    swv::Precomp *sB = reinterpret_cast<swv::Precomp *>(swv_smem);
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.tab + (size_t)a.M * swv::COMB_ENTRIES);
        for (int i = threadIdx.x; i < swv::COMB_ENTRIES * 6; i += blockDim.x) swv_smem[i] = src[i];
    }
    __syncthreads();
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const int i = a.sel ? a.sel[j] : j;
        uint8_t st = 0;
        {
            uint32_t dg[8];
            const int64_t w0 = a.wire_off[i];
            swv::blake2b_256(dg, a.wire + w0, (uint64_t)(a.wire_off[i + 1] - w0));
            const uint32_t *id = reinterpret_cast<const uint32_t *>(a.ids + (size_t)32 * i);
            uint32_t o = 0;
            for (int t = 0; t < 8; t++) o |= dg[t] ^ id[t];
            if (o == 0) st |= 2;
        }
        const int c = a.creator[i];
        if (c >= 0 && c < a.M && a.keyok[c]) {
            const swv::Precomp *tA = a.tab + (size_t)c * swv::COMB_ENTRIES;
            auto tabB = [sB](int e) { return sB[e]; };
            auto tabA = [tA](int e) {
                swv::Precomp q;
                const uint4 *p = reinterpret_cast<const uint4 *>(tA + e);
                uint4 *d = reinterpret_cast<uint4 *>(&q);
#pragma unroll
                for (int t = 0; t < 6; t++) d[t] = __ldg(p + t);
                return q;
            };
            const int64_t m0 = a.msg_off[i];
            if (swv::ed25519_verify(a.sig + (size_t)64 * i, a.pk + (size_t)32 * c, a.msg + m0,
                                    (uint64_t)(a.msg_off[i + 1] - m0), tabB, tabA))
                st |= 1;
        }
        a.status[i] = st;
    }
}
