"""oracle/ecdsa_oracle.py -- ECDSA over P-256 on Python integers (SEC1 v2 section 4.1.4 verification).

TEST INFRASTRUCTURE ONLY: the checker for modarith_b200.ecdsa.  It shares nothing with the product: the curve
constants come from oracle_primes.py, the arithmetic is plain big-integer arithmetic in Jacobian coordinates,
and every decision is an ordinary `if`.  The signer takes its nonce as an argument so that fixtures can be
built with chosen values of R (tests/golden/make_ecdsa_golden.py).
"""
from __future__ import annotations

import oracle_primes

_C = oracle_primes.TABLE["NIST256"]
P = _C.p
N = _C.worder
B = _C.wb
G = (_C.wgx, _C.wgy)
INF = None


def on_curve(pt) -> bool:
    x, y = pt
    return 0 <= x < P and 0 <= y < P and (y * y - (x * x * x - 3 * x + B)) % P == 0


def _jdbl(X, Y, Z):
    if Z == 0 or Y == 0:
        return (1, 1, 0)
    d = Z * Z % P
    g = Y * Y % P
    b = X * g % P
    a = 3 * (X - d) * (X + d) % P
    X3 = (a * a - 8 * b) % P
    Z3 = ((Y + Z) ** 2 - g - d) % P
    Y3 = (a * (4 * b - X3) - 8 * g * g) % P
    return (X3, Y3, Z3)


def _jadd(p1, p2):
    X1, Y1, Z1 = p1
    X2, Y2, Z2 = p2
    if Z1 == 0:
        return p2
    if Z2 == 0:
        return p1
    Z1Z1, Z2Z2 = Z1 * Z1 % P, Z2 * Z2 % P
    U1, U2 = X1 * Z2Z2 % P, X2 * Z1Z1 % P
    S1, S2 = Y1 * Z2 * Z2Z2 % P, Y2 * Z1 * Z1Z1 % P
    if U1 == U2:
        return _jdbl(X1, Y1, Z1) if S1 == S2 else (1, 1, 0)
    H, R = (U2 - U1) % P, (S2 - S1) % P
    HH = H * H % P
    HHH = H * HH % P
    V = U1 * HH % P
    X3 = (R * R - HHH - 2 * V) % P
    Y3 = (R * (V - X3) - S1 * HHH) % P
    return (X3, Y3, Z1 * Z2 * H % P)


def _affine(j):
    X, Y, Z = j
    if Z == 0:
        return INF
    zi = pow(Z, -1, P)
    zi2 = zi * zi % P
    return (X * zi2 % P, Y * zi2 * zi % P)


def _jac(pt):
    return (1, 1, 0) if pt is INF else (pt[0], pt[1], 1)


def add(p1, p2):
    """Affine point addition (INF = the point at infinity)."""
    return _affine(_jadd(_jac(p1), _jac(p2)))


def neg(pt):
    return INF if pt is INF else (pt[0], (-pt[1]) % P)


def mul2(a: int, p1, b: int, p2):
    """a*p1 + b*p2 (Shamir's trick, plain double-and-add)."""
    j1, j2 = _jac(p1), _jac(p2)
    j12 = _jadd(j1, j2)
    acc = (1, 1, 0)
    for i in range(max(a.bit_length(), b.bit_length()) - 1, -1, -1):
        acc = _jdbl(*acc)
        sel = ((a >> i) & 1) | (((b >> i) & 1) << 1)
        if sel:
            acc = _jadd(acc, (j1, j2, j12)[sel - 1])
    return _affine(acc)


def mul(k: int, pt=G):
    return mul2(k, pt, 0, G)


def bits2int(digest: bytes) -> int:
    """The leftmost 256 bits of a digest as an integer (SEC1 v2 4.1.3 step 5)."""
    v = int.from_bytes(digest, "big")
    extra = 8 * len(digest) - 256
    return v >> extra if extra > 0 else v


def verify(h: int, r: int, s: int, q) -> bool:
    """SEC1 v2 4.1.4 with the public-key checks of 3.2.2.1: h = bits2int(digest); q = (x, y) as given."""
    if not (1 <= r < N and 1 <= s < N):
        return False
    if q is INF or not on_curve(q):
        return False
    w = pow(s, -1, N)
    R = mul2(h * w % N, G, r * w % N, q)
    if R is INF:
        return False
    return R[0] % N == r


def sign(d: int, h: int, k: int):
    """(r, s) for private key d, digest integer h and the nonce k; None where r or s would be 0."""
    R = mul(k)
    r = R[0] % N
    s = pow(k, -1, N) * (h + r * d) % N
    if r == 0 or s == 0:
        return None
    return r, s


def public_key(d: int):
    return mul(d)
