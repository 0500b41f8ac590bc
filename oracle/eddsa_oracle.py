"""oracle/eddsa_oracle.py -- Ed25519 on Python integers (RFC 8032 sections 5.1.2-5.1.7, pure Ed25519).

TEST INFRASTRUCTURE ONLY: the checker for modarith_b200.eddsa.  It shares nothing with the product: the curve
constants come from oracle_primes.py, the arithmetic is plain big-integer arithmetic in extended coordinates,
and every decision is an ordinary `if`.  The verification policy is the one the library pins: strict decoding
of A (y < p, a square root, not x = 0 with the sign bit), S < L, k = SHA-512(R || A || M) mod L, the
cofactorless equation encode([S]B - [k]A) == R over all 256 bits, small-order A and R accepted.  Besides the
RFC 8032 signer (from a 32-byte seed) there is a signer with an explicit nonce and secret scalar, so that
fixtures can be built with chosen keys and R (tests/golden/make_eddsa_golden.py).
"""
from __future__ import annotations

import hashlib

import oracle_primes

_C = oracle_primes.TABLE["X25519"]
P = _C.p
D = _C.ed_d
L = _C.ed_order
SQRT_M1 = _C.roi                        # 2^((p-1)/4): a square root of -1 (p = 5 mod 8)
B = (_C.ed_gx, _C.ed_gy)
IDENTITY = (0, 1)


def _ext(pt):
    x, y = pt
    return (x, y, 1, x * y % P)


def _affine(e):
    X, Y, Z, _ = e
    zi = pow(Z, -1, P)
    return (X * zi % P, Y * zi % P)


def _eadd(p1, p2):
    """add-2008-hwcd-3 (a = -1): complete on Ed25519."""
    X1, Y1, Z1, T1 = p1
    X2, Y2, Z2, T2 = p2
    a = (Y1 - X1) * (Y2 - X2) % P
    b = (Y1 + X1) * (Y2 + X2) % P
    c = 2 * D * T1 * T2 % P
    d = 2 * Z1 * Z2 % P
    e, f, g, h = b - a, d - c, d + c, b + a
    return (e * f % P, g * h % P, f * g % P, e * h % P)


def _edbl(p1):
    """dbl-2008-hwcd (a = -1)."""
    X1, Y1, Z1, _ = p1
    a, b = X1 * X1 % P, Y1 * Y1 % P
    c = 2 * Z1 * Z1 % P
    h = a + b
    e = h - (X1 + Y1) ** 2
    g = a - b
    f = c + g
    return (e * f % P, g * h % P, f * g % P, e * h % P)


def add(p1, p2):
    return _affine(_eadd(_ext(p1), _ext(p2)))


def neg(pt):
    return ((-pt[0]) % P, pt[1])


def mul2(a: int, p1, b: int, p2):
    """[a]p1 + [b]p2 (Shamir's trick, plain double-and-add from the top bit)."""
    e1, e2 = _ext(p1), _ext(p2)
    tab = (None, e1, e2, _eadd(e1, e2))
    acc = _ext(IDENTITY)
    for i in range(max(a.bit_length(), b.bit_length()) - 1, -1, -1):
        acc = _edbl(acc)
        sel = ((a >> i) & 1) | (((b >> i) & 1) << 1)
        if sel:
            acc = _eadd(acc, tab[sel])
    return _affine(acc)


def mul(k: int, pt=B):
    return mul2(k, pt, 0, B)


def on_curve(pt) -> bool:
    x, y = pt
    return (-x * x + y * y - 1 - D * x * x * y * y) % P == 0


def encode(pt) -> bytes:
    x, y = pt
    return (y | ((x & 1) << 255)).to_bytes(32, "little")


def recover_x(y: int, sign: int):
    """x with x^2 = (y^2 - 1)/(d y^2 + 1) and the given low bit, or None (no root, or x = 0 with sign 1)."""
    u, v = (y * y - 1) % P, (D * y * y + 1) % P
    x2 = u * pow(v, -1, P) % P
    x = pow(x2, (P + 3) // 8, P)
    if (x * x - x2) % P != 0:
        x = x * SQRT_M1 % P
    if (x * x - x2) % P != 0:
        return None
    if x == 0 and sign:
        return None
    if x & 1 != sign:
        x = P - x
    return x


def decode(enc: bytes):
    """RFC 8032 5.1.3, strict: the point, or None (wrong length, y >= p, no root, x = 0 with the sign bit)."""
    if len(enc) != 32:
        return None
    v = int.from_bytes(enc, "little")
    y, sign = v & ((1 << 255) - 1), v >> 255
    if y >= P:
        return None
    x = recover_x(y, sign)
    return None if x is None else (x, y)


def digest(R: bytes, A: bytes, msg: bytes) -> bytes:
    return hashlib.sha512(bytes(R) + bytes(A) + bytes(msg)).digest()


def verify_digest(h: bytes, sig: bytes, A: bytes) -> bool:
    """The library's policy on h = SHA-512(R || A || M), sig = R || S and the encoded key A."""
    if len(h) != 64 or len(sig) != 64 or len(A) != 32:
        return False
    R, S = bytes(sig[:32]), int.from_bytes(sig[32:], "little")
    if S >= L:
        return False
    a = decode(A)
    if a is None:
        return False
    k = int.from_bytes(h, "little") % L
    return encode(mul2(S, B, k, neg(a))) == R


def verify(msg: bytes, sig: bytes, A: bytes) -> bool:
    if len(sig) != 64 or len(A) != 32:
        return False
    return verify_digest(digest(sig[:32], A, msg), sig, A)


def secret_scalar(seed: bytes):
    """(a, prefix) of RFC 8032 5.1.5 for a 32-byte seed."""
    hs = hashlib.sha512(seed).digest()
    a = int.from_bytes(hs[:32], "little")
    a &= (1 << 254) - 8
    a |= 1 << 254
    return a, hs[32:]


def public_key(seed: bytes) -> bytes:
    return encode(mul(secret_scalar(seed)[0]))


def sign(seed: bytes, msg: bytes) -> bytes:
    """RFC 8032 5.1.6."""
    a, prefix = secret_scalar(seed)
    A = encode(mul(a))
    r = int.from_bytes(hashlib.sha512(prefix + bytes(msg)).digest(), "little") % L
    return sign_with_nonce(a, r, msg, A)


def sign_with_nonce(a: int, r: int, msg: bytes, A: bytes) -> bytes:
    """R || S with R = [r]B and S = r + k a mod L, k = SHA-512(R || A || M) mod L, for any encoding A (also one
    that is not [a]B: the result then verifies only where the equation happens to hold)."""
    R = encode(mul(r))
    k = int.from_bytes(digest(R, A, msg), "little") % L
    return R + ((r + k * a) % L).to_bytes(32, "little")
