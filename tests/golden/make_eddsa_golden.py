#!/usr/bin/env python3
"""Write tests/golden/eddsa_ed25519_sample.json in the Wycheproof layout (eddsa_verify_schema: testGroups[] of type
EddsaVerify with publicKey.curve / publicKey.pk, tests[] with tcId, comment, flags, msg, sig, result).  Seeded: the
same file on every run.

Every row's `result` is the library's policy (RFC 8032 5.1.7 with strict decoding of A, S < L, the cofactorless
equation, small-order A and R accepted), computed by oracle/eddsa_oracle.py; the script asserts that it is the result
each row was built to have.  OpenSSL (through `cryptography`) agrees on every row except the ones flagged
"NonCanonicalPublicKey": keys whose y is given as y + p, or x = 0 with the sign bit set, which OpenSSL decodes
leniently and accepts where the equation holds.  The script asserts that too.

The rows: honest signatures (random, RFC 8032 7.1 TEST 1 and TEST 2, empty and 1 KiB messages); S + L; the
identity key (canonical, as y = p + 1, as (0, 1) with the sign bit); a key with an order-8 component with k = 0 and
k != 0 mod 8; S = L - 1, L, 2^255 - 1, 2^256 - 1 and 2^255; every y < 19 whose encoding y + p decodes, both sign bits;
a y with no square root; y = p - 1 with the sign bit; a non-canonical R; R with its sign bit flipped; small-order R;
wrong message, wrong key; signatures of 63 and 65 bytes and a 31-byte key.

    python tests/golden/make_eddsa_golden.py
"""
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import eddsa_oracle as O  # noqa: E402

from cryptography.exceptions import InvalidSignature  # noqa: E402
from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PublicKey  # noqa: E402

P, L = O.P, O.L
FLAG = "NonCanonicalPublicKey"
rng = random.Random(0xED25519)
le = lambda v: (v % (1 << 256)).to_bytes(32, "little")


def openssl(msg, sig, pk):
    try:
        Ed25519PublicKey.from_public_bytes(pk).verify(sig, msg)
        return True
    except (InvalidSignature, ValueError):
        return False


def order8_point():
    """A point of order exactly 8: [L] of the first decodable y >= 2 whose torsion part has order 8."""
    for y in range(2, 1000):
        x = O.recover_x(y, 0)
        if x is None:
            continue
        t = O.mul(L, (x, y))
        if O.mul(4, t) != O.IDENTITY:
            return t
    raise AssertionError("no order-8 point found")


def seed_key():
    seed = rng.randbytes(32)
    return seed, O.public_key(seed)


def r_of_sb(A, order, msg_prefix):
    """(msg, S, R) with R = enc([S]B) and k = H(R || A || M) = 0 mod `order`: valid under any verifier that decodes
    A to a point of that order (then [k]A = O)."""
    while True:
        S = rng.randrange(L)
        R = O.encode(O.mul(S))
        msg = msg_prefix + rng.randbytes(8)
        if int.from_bytes(O.digest(R, A, msg), "little") % L % order == 0:
            return msg, R + le(S)


rows = []        # (comment, pk bytes, msg, sig, intended validity)


def add(comment, pk, msg, sig, valid):
    rows.append((comment, bytes(pk), bytes(msg), bytes(sig), valid))


# honest signatures, RFC 8032 7.1
for i in range(6):
    seed, pk = seed_key()
    msg = rng.randbytes(rng.randrange(1, 100))
    add("honest signature", pk, msg, O.sign(seed, msg), True)
T1 = ("9d61b19deffd5a60ba844af492ec2cc44449c5697b326919703bac031cae7f60",
      "d75a980182b10ab7d54bfed3c964073a0ee172f3daa62325af021a68f707511a", "",
      "e5564300c360ac729086e2cc806e828a84877f1eb8e5d974d873e065224901555fb8821590a33bacc61e39701cf9b46bd25bf5f0595bbe24655141438e7a100b")
T2 = ("4ccd089b28ff96da9db6c346ec114e0f5b8a319f35aba624da8cf6ed4fb8a6fb",
      "3d4017c3e843895a92b70aa74d1b7ebc9c982ccf2ec4968cc0cd55f12af4660c", "72",
      "92a009a9f0d4cab8720e820b5f642540a2b27b5416503f8fb3762223ebdb69da085ac1e43e15996e458f3613d0f11d8c387b2eaeb4302aeeb00d291612bb0c00")
for name, (sk, pk, msg, sig) in (("RFC 8032 7.1 TEST 1", T1), ("RFC 8032 7.1 TEST 2", T2)):
    assert O.public_key(bytes.fromhex(sk)).hex() == pk and O.sign(bytes.fromhex(sk), bytes.fromhex(msg)).hex() == sig
    add(name, bytes.fromhex(pk), bytes.fromhex(msg), bytes.fromhex(sig), True)
seed, pk = seed_key()
add("empty message", pk, b"", O.sign(seed, b""), True)
msg = rng.randbytes(1024)
add("1 KiB message", pk, msg, O.sign(seed, msg), True)

# S + L (malleability)
seed, pk = seed_key()
msg = rng.randbytes(20)
sig = O.sign(seed, msg)
add("S replaced by S + L", pk, msg, sig[:32] + le(int.from_bytes(sig[32:], "little") + L), False)

# identity key: canonical, as y = p + 1, as (0, 1) with the sign bit
ID = le(1)
msg, sig = r_of_sb(ID, 1, b"id")
add("A = identity, R = enc([S]B)", ID, msg, sig, True)
NC_ID = le(P + 1)
msg, sig = r_of_sb(NC_ID, 1, b"id")
add("A = identity as y = p + 1 (non-canonical)", NC_ID, msg, sig, False)
SIGNED_ID = le(1 | (1 << 255))
msg, sig = r_of_sb(SIGNED_ID, 1, b"id")
add("A = (0, 1) with the sign bit set", SIGNED_ID, msg, sig, False)

# A = aB + T8, honest signature under that encoding
T8 = order8_point()
a = rng.randrange(1, L)
A8 = O.encode(O.add(O.mul(a), T8))
done = set()
while len(done) < 2:
    msg = rng.randbytes(16)
    sig = O.sign_with_nonce(a, rng.randrange(1, L), msg, A8)
    k = int.from_bytes(O.digest(sig[:32], A8, msg), "little") % L
    kind = k % 8 == 0
    if kind in done:
        continue
    done.add(kind)
    add("A = aB + T8, k = 0 mod 8" if kind else "A = aB + T8, k != 0 mod 8 (a cofactored verifier would accept)",
        A8, msg, sig, kind)

# S range edges under the identity key: R = enc([S mod L]B), so only the S < L check decides
for name, S in (("S = L - 1", L - 1), ("S = L", L), ("S = 2^255 - 1", (1 << 255) - 1), ("S = 2^256 - 1", (1 << 256) - 1),
                ("S = 2^255 (only bit 255 set)", 1 << 255)):
    add(name, ID, b"S edge", O.encode(O.mul(S % L)) + le(S), S < L)

# non-canonical y: y + p for y < 19 where it decodes, both sign bits
for y in range(19):
    for sign in (0, 1):
        if y > 1 and O.recover_x(y, sign) is None:
            continue
        if y <= 1 and O.recover_x(y, 0) is None:
            continue
        enc = le((y + P) | (sign << 255))
        order = 1 if y == 1 else 4 if y == 0 else None           # (0, 1) is O; y = 0 is a point of order 4
        if order:
            msg, sig = r_of_sb(enc, order, b"nc")
        else:
            msg = rng.randbytes(12)
            S = rng.randrange(L)
            sig = O.encode(O.mul(S)) + le(S)
        add("non-canonical key y = %d + p, sign %d" % (y, sign), enc, msg, sig, False)
# a y with no square root
y = next(y for y in range(2, 100) if O.recover_x(y, 0) is None)
enc = le(y)
msg, sig = r_of_sb(enc, 1, b"ns")
add("key y = %d has no square root" % y, enc, msg, sig, False)
# y = p - 1 with the sign bit: x = 0, a point of order 2
enc = le((P - 1) | (1 << 255))
msg, sig = r_of_sb(enc, 2, b"pm1")
add("key y = p - 1 with the sign bit (x = 0)", enc, msg, sig, False)

# R: non-canonical, sign bit flipped, small order
add("non-canonical R: the identity as y = p + 1", ID, b"R", le(P + 1) + le(0), False)
add("R = identity (small order), S = 0, A = identity", ID, b"R", le(1) + le(0), True)
T2P = le(P - 1)                                                 # (0, -1): order 2, canonical encoding
while True:
    msg = b"R2" + rng.randbytes(8)
    if int.from_bytes(O.digest(T2P, T2P, msg), "little") % L % 2 == 1:
        break
add("R of order 2, S = 0, A of order 2", T2P, msg, T2P + le(0), True)
seed, pk = seed_key()
msg = rng.randbytes(20)
sig = O.sign(seed, msg)
add("R with its sign bit flipped", pk, msg, sig[:31] + bytes([sig[31] ^ 0x80]) + sig[32:], False)

# wrong message, wrong key, lengths
seed, pk = seed_key()
_, pk2 = seed_key()
msg = rng.randbytes(20)
sig = O.sign(seed, msg)
add("wrong message", pk, msg + b"\x00", sig, False)
add("wrong key", pk2, msg, sig, False)
add("signature of 63 bytes", pk, msg, sig[:63], False)
add("signature of 65 bytes", pk, msg, sig + b"\x00", False)
add("key of 31 bytes", pk[:31], msg, sig, False)

groups, tc = [], 0
for comment, pk, msg, sig, valid in rows:
    ours = O.verify(msg, sig, pk)
    assert ours == valid, comment
    theirs = openssl(msg, sig, pk)
    flags = []
    if theirs != ours:
        noncanonical = len(pk) == 32 and ((int.from_bytes(pk, "little") & ((1 << 255) - 1)) >= P or
                                          (pk[31] >> 7 and O.recover_x(int.from_bytes(pk, "little") % (1 << 255) % P, 0) == 0))
        assert noncanonical and theirs and not ours, comment
        flags = [FLAG]
    tc += 1
    test = {"tcId": tc, "comment": comment, "flags": flags, "msg": msg.hex(), "sig": sig.hex(),
            "result": "valid" if valid else "invalid"}
    if groups and groups[-1]["publicKey"]["pk"] == pk.hex():
        groups[-1]["tests"].append(test)
    else:
        groups.append({"type": "EddsaVerify",
                       "publicKey": {"type": "EDDSAPublicKey", "curve": "edwards25519", "keySize": 255, "pk": pk.hex()},
                       "tests": [test]})
doc = {"algorithm": "EDDSA", "numberOfTests": tc,
       "header": ["Ed25519 verification edge cases, generated by tests/golden/make_eddsa_golden.py.",
                  "result is the policy of modarith_b200.eddsa (RFC 8032 5.1.7, strict key decoding, S < L,",
                  "cofactorless equation); OpenSSL agrees except on rows flagged %s." % FLAG],
       "notes": {FLAG: "the key's y is given as y + p, or x = 0 with the sign bit set; OpenSSL decodes it leniently "
                       "and accepts, RFC 8032 5.1.3 decoding (and this library) rejects"},
       "schema": "eddsa_verify_schema.json", "testGroups": groups}
out = os.path.join(HERE, "eddsa_ed25519_sample.json")
# one test per line: the file stays readable and small in a diff
text = json.dumps(doc, indent=1)
for g in groups:
    for t in g["tests"]:
        text = text.replace(json.dumps(t, indent=1).replace("\n", "\n    "), json.dumps(t), 1)
assert json.loads(text) == doc
with open(out, "w") as f:
    f.write(text + "\n")
print("wrote", out, tc, "tests,", sum(1 for r in rows if r[4]), "valid,",
      sum(1 for g in groups for t in g["tests"] if t["flags"]), "flagged")
