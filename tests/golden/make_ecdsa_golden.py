#!/usr/bin/env python3
"""Write tests/golden/ecdsa_secp256r1_sha256_sample.json (DER signatures) and its twin
ecdsa_secp256r1_sha256_p1363_sample.json (r || s) in the Wycheproof layout (ecdsa_verify_schema /
ecdsa_p1363_verify_schema: testGroups[] with publicKey.uncompressed, sha, tests[] with tcId, comment, flags, msg,
sig, result).  Seeded: the same files on every run.

Every row's `result` is what BOTH oracle/ecdsa_oracle.py (SEC1 v2 4.1.4 on integers, signatures decoded with
cryptography's decode_dss_signature) and OpenSSL (through `cryptography`) say; the script asserts they agree.

The rows: valid signatures and their s -> n - s twins; r or s in {0, n, n + 1, 2^256 - 1} and r = s = 1; digests 0, n
and 2^256 - 1; h = -r d (u1 G + u2 Q = O); a valid signature whose x(R) lies in [n, p) (the r + n case), and the
same with the unreduced x(R) as r; r = p - n - 1 and r = p - n; keys off the curve, with x given as x + p, Q = G
and Q = -G; malformed DER (long-form and non-minimal lengths, padded and negative INTEGERs, trailing bytes, a
missing s, 33- and 34-byte integers, indefinite length) or P1363 strings of the wrong length.

Rows that need a chosen digest sit in groups marked `"prehashed": true`, whose `msg` is the 32-byte digest itself
(modarith_b200.wire.load_ecdsa_vectors; OpenSSL checks them with Prehashed(SHA256())).

    python tests/golden/make_ecdsa_golden.py
"""
import hashlib
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import ecdsa_oracle as O  # noqa: E402

from cryptography.exceptions import InvalidSignature  # noqa: E402
from cryptography.hazmat.primitives import hashes  # noqa: E402
from cryptography.hazmat.primitives.asymmetric import ec, utils  # noqa: E402

N, P = O.N, O.P
rng = random.Random(0xEC05A)


def be(v, nb=32):
    return v.to_bytes(nb, "big")


def der_int(v, pad=0):
    b = v.to_bytes(max(1, (v.bit_length() + 7) // 8), "big")
    if b[0] & 0x80:
        b = b"\x00" + b
    return b"\x00" * pad + b


def der_tlv(tag, body, long_form=False):
    if long_form or len(body) >= 0x80:
        return bytes([tag, 0x81, len(body)]) + body
    return bytes([tag, len(body)]) + body


def der(r, s):
    return der_tlv(0x30, der_tlv(0x02, der_int(r)) + der_tlv(0x02, der_int(s)))


def key_hex(q):
    return (b"\x04" + be(q[0]) + be(q[1])).hex()


def sqrt_p(v):
    y = pow(v, (P + 1) // 4, P)
    return y if y * y % P == v % P else None


def digest(msg, prehashed):
    return msg if prehashed else hashlib.sha256(msg).digest()


def openssl(key, sig, msg, prehashed, encoding):
    try:
        pk = ec.EllipticCurvePublicKey.from_encoded_point(ec.SECP256R1(), key)
    except ValueError:
        return False
    if encoding == "p1363":
        if len(sig) != 64:
            return False
        sig = utils.encode_dss_signature(int.from_bytes(sig[:32], "big"), int.from_bytes(sig[32:], "big"))
    algo = ec.ECDSA(utils.Prehashed(hashes.SHA256()) if prehashed else hashes.SHA256())
    try:
        pk.verify(sig, msg, algo)
        return True
    except InvalidSignature:
        return False


def oracle(key, sig, msg, prehashed, encoding):
    if len(key) != 65 or key[0] != 4:
        return False
    q = (int.from_bytes(key[1:33], "big"), int.from_bytes(key[33:], "big"))
    if encoding == "p1363":
        if len(sig) != 64:
            return False
        r, s = int.from_bytes(sig[:32], "big"), int.from_bytes(sig[32:], "big")
    else:
        try:
            r, s = utils.decode_dss_signature(sig)
        except ValueError:
            return False
    return O.verify(O.bits2int(digest(msg, prehashed)), r, s, q)


class Group:
    def __init__(self, key, prehashed=False):
        self.key, self.prehashed, self.rows = key, prehashed, []

    def add(self, comment, msg, r, s, der_sig=None, p1363_sig=None, flags=()):
        """r, s: the integers, encoded either way; or None with an explicit string for one encoding only."""
        self.rows.append((comment, msg, r, s, der_sig, p1363_sig, list(flags)))


def signed(d, msg, prehashed=False, k=None):
    h = O.bits2int(digest(msg, prehashed))
    while True:
        rs = O.sign(d, h, k or rng.randrange(1, N))
        if rs:
            return rs
        k = None


def build_groups():
    groups = []
    d = rng.randrange(1, N)
    Q = O.public_key(d)
    g = Group(Q)
    for i in range(6):
        msg = bytes(rng.randrange(256) for _ in range(rng.randrange(0, 40)))
        r, s = signed(d, msg)
        g.add("valid signature %d" % i, msg, r, s, flags=["Valid"])
        g.add("valid signature %d with s -> n - s" % i, msg, r, N - s, flags=["Valid", "SignatureMalleability"])
    msg = b"123400"
    r0, s0 = signed(d, msg)
    g.add("valid reference signature", msg, r0, s0, flags=["Valid"])
    for v, name in ((0, "0"), (N, "n"), (N + 1, "n + 1"), ((1 << 256) - 1, "2^256 - 1")):
        g.add("r = %s" % name, msg, v, s0, flags=["RangeCheck"])
        g.add("s = %s" % name, msg, r0, v, flags=["RangeCheck"])
    g.add("r = s = 1", msg, 1, 1, flags=["RangeCheck"])
    g.add("r = p - n - 1", msg, P - N - 1, s0, flags=["ArithmeticError"])
    g.add("r = p - n", msg, P - N, s0, flags=["ArithmeticError"])
    g.add("r + 1", msg, r0 + 1, s0, flags=["ModifiedSignature"])
    g.add("wrong message", b"123401", r0, s0, flags=["ModifiedSignature"])
    # malformed DER of the reference signature (P1363 twins: strings of the wrong length)
    ir, is_ = der_tlv(0x02, der_int(r0)), der_tlv(0x02, der_int(s0))
    rb = r0.to_bytes(32, "big")
    bad = [
        ("long-form SEQUENCE length", der_tlv(0x30, ir + is_, long_form=True)),
        ("long-form INTEGER length", der_tlv(0x30, der_tlv(0x02, der_int(r0), long_form=True) + is_)),
        ("non-minimal SEQUENCE length (0x82)", bytes([0x30, 0x82, 0x00, len(ir + is_)]) + ir + is_),
        ("INTEGER padded with 0x00", der_tlv(0x30, der_tlv(0x02, der_int(r0, pad=1)) + is_)),
        ("negative INTEGER", der_tlv(0x30, der_tlv(0x02, bytes([rb[0] | 0x80]) + rb[1:]) + is_)),
        ("trailing byte after the SEQUENCE", der(r0, s0) + b"\x00"),
        ("trailing byte inside the SEQUENCE", der_tlv(0x30, ir + is_ + b"\x00")),
        ("missing s", der_tlv(0x30, ir)),
        ("33-byte INTEGER r + 2^256", der_tlv(0x30, der_tlv(0x02, der_int(r0 + (1 << 256))) + is_)),
        ("34-byte INTEGER (two leading zeros)", der_tlv(0x30, der_tlv(0x02, b"\x00\x00" + rb) + is_)),
        ("indefinite length", b"\x30\x80" + ir + is_ + b"\x00\x00"),
        ("empty INTEGER", der_tlv(0x30, b"\x02\x00" + is_)),
        ("wrong tag", der_tlv(0x31, ir + is_)),
        ("empty signature", b""),
    ]
    for name, sig in bad:
        g.add("DER: " + name, msg, None, None, der_sig=sig, flags=["InvalidEncoding"])
    rs = be(r0) + be(s0)
    for name, sig in (("63 bytes", rs[:63]), ("65 bytes", rs + b"\x00"), ("empty", b""), ("r only", rs[:32])):
        g.add("P1363: " + name, msg, None, None, p1363_sig=sig, flags=["InvalidEncoding"])
    groups.append(g)

    # chosen digests: 0, n, 2^256 - 1, and h = -r d (u1 G + u2 Q = O)
    g = Group(Q, prehashed=True)
    for v, name in ((0, "0"), (N, "n"), ((1 << 256) - 1, "2^256 - 1")):
        r, s = signed(d, be(v), prehashed=True)
        g.add("digest %s" % name, be(v), r, s, flags=["Valid"])
        g.add("digest %s, s + 1" % name, be(v), r, s + 1, flags=["ModifiedSignature"])
    r, s = r0, s0
    g.add("h = -r d: u1 G + u2 Q = O", be((-r * d) % N), r, s, flags=["PointAtInfinity"])
    groups.append(g)

    # x(R) in [n, p): r = x(R) - n, key Q = u2^-1 (R - u1 G)
    t = 0
    while True:
        x = N + t
        y = sqrt_p((x * x * x - 3 * x + O.B) % P)
        if y is not None and x < P:
            break
        t += 1
    Rpt = (x, y)
    msg = b"x(R) >= n"
    h = O.bits2int(digest(msg, False))
    r = x - N
    s = rng.randrange(1, N)
    w = pow(s, -1, N)
    u1, u2 = h * w % N, r * w % N
    Qx = O.mul(pow(u2, -1, N), O.add(Rpt, O.neg(O.mul(u1))))
    g = Group(Qx)
    g.add("x(R) in [n, p): r = x(R) - n", msg, r, s, flags=["ArithmeticError"])
    g.add("x(R) in [n, p): r = x(R) unreduced", msg, x, s, flags=["RangeCheck"])
    groups.append(g)

    # keys: Q = G, Q = -G, off the curve, x given as x + p
    for dd, name in ((1, "Q = G"), (N - 1, "Q = -G")):
        g = Group(O.public_key(dd))
        r, s = signed(dd, b"generator")
        g.add(name, b"generator", r, s, flags=["Valid"])
        groups.append(g)
    g = Group((Q[0], (Q[1] + 1) % P))
    g.add("public key off the curve", b"123400", r0, s0, flags=["InvalidPublicKey"])
    groups.append(g)
    xs = 0
    while sqrt_p((xs ** 3 - 3 * xs + O.B) % P) is None or xs + P >= 1 << 256:
        xs += 1
    Qs = (xs, sqrt_p((xs ** 3 - 3 * xs + O.B) % P))
    u1, u2 = rng.randrange(1, N), rng.randrange(1, N)
    Rpt = O.mul2(u1, O.G, u2, Qs)
    r = Rpt[0] % N
    w = u2 * pow(r, -1, N) % N
    s, h = pow(w, -1, N), u1 * pow(w, -1, N) % N
    assert O.verify(h, r, s, Qs)
    g = Group(Qs, prehashed=True)
    g.add("small x, key as given (valid)", be(h), r, s, flags=["Valid"])
    groups.append(g)
    g = Group((xs + P, Qs[1]), prehashed=True)
    g.add("key coordinate x + p", be(h), r, s, flags=["InvalidPublicKey"])
    groups.append(g)
    return groups


def write(groups, encoding, path):
    tc = 0
    out_groups = []
    nvalid = 0
    for g in groups:
        tests = []
        for comment, msg, r, s, der_sig, p_sig, flags in g.rows:
            if encoding == "der":
                if der_sig is None and r is None:
                    continue
                sig = der_sig if der_sig is not None else der(r, s)
            else:
                if p_sig is None and (r is None or r >= 1 << 256 or s >= 1 << 256):
                    continue
                sig = p_sig if p_sig is not None else be(r) + be(s)
            key = b"\x04" + be(g.key[0]) + be(g.key[1])
            a, b = oracle(key, sig, msg, g.prehashed, encoding), openssl(key, sig, msg, g.prehashed, encoding)
            assert a == b, (comment, encoding, a, b)
            tc += 1
            nvalid += a
            tests.append({"tcId": tc, "comment": comment, "flags": flags, "msg": msg.hex(), "sig": sig.hex(),
                          "result": "valid" if a else "invalid"})
        grp = {"type": "EcdsaVerify" if encoding == "der" else "EcdsaP1363Verify",
               "publicKey": {"type": "EcPublicKey", "curve": "secp256r1", "keySize": 256,
                             "uncompressed": key_hex(g.key), "wx": be(g.key[0]).hex(), "wy": be(g.key[1]).hex()},
               "sha": "SHA-256"}
        if g.prehashed:
            grp["prehashed"] = True
        grp["tests"] = tests
        out_groups.append(grp)
    doc = {"algorithm": "ECDSA", "schema": "ecdsa_verify_schema.json" if encoding == "der" else "ecdsa_p1363_verify_schema.json",
           "numberOfTests": tc,
           "header": ["Edge cases of ECDSA P-256 verification, generated by tests/golden/make_ecdsa_golden.py;",
                      "every result agreed by oracle/ecdsa_oracle.py and OpenSSL."],
           "notes": {}, "testGroups": out_groups}
    with open(path, "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")
    print("wrote %s: %d tests, %d valid" % (path, tc, nvalid))


if __name__ == "__main__":
    gs = build_groups()
    write(gs, "der", os.path.join(HERE, "ecdsa_secp256r1_sha256_sample.json"))
    write(gs, "p1363", os.path.join(HERE, "ecdsa_secp256r1_sha256_p1363_sample.json"))
