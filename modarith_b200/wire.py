"""Wire and file formats around the batch API (SURVEY.md section 8(f) row 4).

Counterpart of the reference's hex/byte helpers (`rfc7748.c:44-107`) and of its Wycheproof
converter (`parse.py`), restated for batches:

* `from_hex`, `to_hex`, `reverse` take / return `[n, Nbytes]` uint8 arrays instead of one
  `char[Nbytes]`, with `fromHex`'s conventions: a short string is padded with leading zeros, a
  long one is cut after 2*Nbytes characters, a character that is not a hex digit counts as 0
  (`char2int`, rfc7748.c:44-53), output is lower case (`byte2hex`, rfc7748.c:55-67).
* `parse_signature_vectors` is `parse.py`'s scan of a Wycheproof ECDSA/EdDSA file (public key,
  comment, message, signature, outcome per test, in file order) returned as records instead of
  printed lines; `signature_lines` prints them exactly as `parse.py` does.
* `load_xdh_vectors` / `run_xdh_vectors` read a Wycheproof XDH file (`x25519_test.json`,
  `x448_test.json`: `testGroups[].tests[]` with `public`, `private`, `shared`, `result`) into the
  byte arrays `rfc7748()` takes and push the whole suite through the batch ladder in one call --
  the "external vector suites through the batch API" use the survey names.
* `load_ecdsa_vectors` / `run_ecdsa_vectors` do the same for Wycheproof ECDSA verification files
  (`EcdsaVerify` groups with DER signatures, `EcdsaP1363Verify` groups with r || s; secp256r1 only) through
  `modarith_b200.ecdsa`.
* `load_eddsa_vectors` / `run_eddsa_vectors` do the same for Wycheproof EdDSA verification files (`EddsaVerify`
  groups on edwards25519) through `modarith_b200.eddsa`.

Host-side format code only: nothing here computes field arithmetic.
"""
from __future__ import annotations

import json
from dataclasses import dataclass
from typing import Iterable, List, Sequence

import numpy as np

__all__ = ["from_hex", "to_hex", "reverse", "parse_signature_vectors", "signature_lines",
           "SignatureVector", "XdhVector", "load_xdh_vectors", "run_xdh_vectors", "EcdsaVector", "load_ecdsa_vectors",
           "run_ecdsa_vectors", "EddsaVector", "load_eddsa_vectors", "run_eddsa_vectors"]

_HEXVAL = np.zeros(256, dtype=np.uint8)
for _c in range(256):
    ch = chr(_c)
    if "0" <= ch <= "9":
        _HEXVAL[_c] = _c - ord("0")
    elif "A" <= ch <= "F":
        _HEXVAL[_c] = _c - ord("A") + 10
    elif "a" <= ch <= "f":
        _HEXVAL[_c] = _c - ord("a") + 10
_HEXDIG = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)


def from_hex(strings: Sequence[str], nbytes: int) -> np.ndarray:
    """`fromHex` (rfc7748.c:81-97) for a batch: [n, nbytes] uint8, big-endian as written."""
    n = len(strings)
    txt = np.full((n, 2 * nbytes), ord("0"), dtype=np.uint8)
    for i, s in enumerate(strings):
        b = s.encode("latin-1", "replace")[: 2 * nbytes]     # a longer string keeps its first 2*Nbytes characters
        if b:
            txt[i, 2 * nbytes - len(b):] = np.frombuffer(b, dtype=np.uint8)
    v = _HEXVAL[txt]
    return ((v[:, 0::2] << 4) | v[:, 1::2]).astype(np.uint8)


def to_hex(data) -> List[str]:
    """`toHex` (rfc7748.c:70-78) for a batch: one lower-case string of 2*Nbytes digits per row."""
    a = np.ascontiguousarray(np.asarray(data, dtype=np.uint8))
    if a.ndim == 1:
        a = a[None, :]
    out = np.empty((a.shape[0], 2 * a.shape[1]), dtype=np.uint8)
    out[:, 0::2] = _HEXDIG[a >> 4]
    out[:, 1::2] = _HEXDIG[a & 15]
    return [row.tobytes().decode("ascii") for row in out]


def reverse(data) -> np.ndarray:
    """`reverse` (rfc7748.c:100-107): byte order of every row flipped (little <-> big endian)."""
    a = np.asarray(data, dtype=np.uint8)
    return np.ascontiguousarray(a[..., ::-1])


# ---------------------------------------------------------------------------------------------
# parse.py: signature suites
# ---------------------------------------------------------------------------------------------
@dataclass
class SignatureVector:
    public_key: str
    comment: str
    msg: str
    sig: str
    result: str


def _extract(s: str, ptr: int, ident: str):
    """`extract` of parse.py:9-13: the quoted string that follows `ident` at or after `ptr`."""
    pk = s.find(ident, ptr)
    fpk = s.find('"', pk + len(ident))
    lpk = s.find('"', fpk + 1) + 1
    return s[fpk + 1:lpk - 1], lpk


def parse_signature_vectors(text: str, kind: str) -> List[SignatureVector]:
    """parse.py:15-52.  `kind` is what parse.py derives from the file name: "ecdsa" (public key
    field `"uncompressed"`) or "ed" (`"pk"`).  The scan is textual, like the reference's, so the
    records come out in file order with the enclosing group's public key attached."""
    if kind.startswith("ecdsa"):
        pubkey = '"uncompressed"'
    elif kind.startswith("ed"):
        pubkey = '"pk"'
    else:
        raise ValueError("parse.py handles ecdsa*/ed* files only")
    out: List[SignatureVector] = []
    ptr = 0
    finished = text.find(pubkey) < 0
    while not finished:
        pk, ptr = _extract(text, ptr, pubkey)
        npk = text.find(pubkey, ptr)
        if npk < 0:
            npk = len(text)
        while True:
            comment, ptr = _extract(text, ptr, '"comment"')
            msg, ptr = _extract(text, ptr, '"msg"')
            sig, ptr = _extract(text, ptr, '"sig"')
            result, ptr = _extract(text, ptr, '"result"')
            out.append(SignatureVector(pk, comment, msg, sig, result))
            nmg = text.find('"comment"', ptr)
            if nmg < 0:
                finished = True
                break
            if nmg >= npk:
                break
    return out


def signature_lines(vectors: Iterable[SignatureVector]) -> str:
    """The five lines per test that parse.py prints (public key, comment, message, signature, outcome)."""
    rows = []
    for v in vectors:
        rows += [v.public_key, v.comment, v.msg, v.sig, v.result]
    return "".join(r + "\n" for r in rows)


# ---------------------------------------------------------------------------------------------
# XDH suites through the batch ladder
# ---------------------------------------------------------------------------------------------
@dataclass
class XdhVector:
    tc_id: int
    comment: str
    public: str
    private: str
    shared: str
    result: str
    flags: tuple


def load_xdh_vectors(source) -> List[XdhVector]:
    """Wycheproof XDH schema (xdh_comp_schema): accepts a path, JSON text or a parsed dict."""
    if isinstance(source, dict):
        doc = source
    else:
        s = str(source)
        doc = json.loads(s) if s.lstrip().startswith("{") else json.load(open(s))
    out = []
    for g in doc.get("testGroups", []):
        for t in g.get("tests", []):
            out.append(XdhVector(int(t.get("tcId", len(out) + 1)), t.get("comment", ""), t["public"], t["private"],
                                 t["shared"], t.get("result", "valid"), tuple(t.get("flags", ()))))
    return out


def run_xdh_vectors(curve: str, vectors: Sequence[XdhVector], device=None):
    """All vectors of a suite in ONE batch call of the ladder (`modarith_b200.rfc7748.rfc7748`).

    Wycheproof writes keys as the raw little-endian RFC 7748 strings, i.e. exactly the `bk`/`bu`
    byte strings (the reference's main feeds the RFC's hex to fromHex the same way, rfc7748.c:271-280).  A test
    passes when the computed string equals `shared`; "invalid" tests must differ or, for XDH,
    usually name the all-zero output, which a caller treats as a failed exchange (RFC 7748 section
    6.1).  Returns (computed [n, Nbytes] uint8, passed bool[n])."""
    from .primes import PRIMES
    from .rfc7748 import rfc7748

    nb = PRIMES[curve].nbytes
    good = [v for v in vectors if len(v.private) == 2 * nb and len(v.public) == 2 * nb]
    bk = from_hex([v.private for v in good], nb)
    bu = from_hex([v.public for v in good], nb)
    bv = rfc7748(curve, bk, bu, device=device) if good else np.zeros((0, nb), dtype=np.uint8)
    bv = bv.cpu().numpy() if hasattr(bv, "cpu") else np.asarray(bv)
    want = from_hex([v.shared for v in good], nb)
    same = (bv == want).all(axis=1)
    zero = (bv == 0).all(axis=1)
    passed = np.empty(len(vectors), dtype=bool)
    gi = 0
    for i, v in enumerate(vectors):
        if len(v.private) != 2 * nb or len(v.public) != 2 * nb:
            passed[i] = v.result != "valid"            # wrong-length keys never reach the ladder
            continue
        if v.result == "invalid":
            passed[i] = bool(zero[gi] or not same[gi])
        else:                                          # "valid" and "acceptable" both pin the shared secret
            passed[i] = bool(same[gi])
        gi += 1
    return bv, passed


# ---------------------------------------------------------------------------------------------
# ECDSA P-256 suites through the batch verifier
# ---------------------------------------------------------------------------------------------
@dataclass
class EcdsaVector:
    tc_id: int
    comment: str
    msg: str
    sig: str
    result: str
    flags: tuple
    public_key: str          # SEC1 uncompressed, hex
    hash: str                # hashlib name; None when `msg` is the digest itself (groups marked "prehashed")
    encoding: str            # "der" or "p1363"


_ECDSA_GROUPS = {"EcdsaVerify": "der", "EcdsaP1363Verify": "p1363"}


def _hashlib_name(sha: str) -> str:
    """Wycheproof's "SHA-256", "SHA3-256", "SHA-512/256" -> hashlib's "sha256", "sha3_256", "sha512_256"."""
    return sha.lower().replace("sha3-", "sha3_").replace("/", "_").replace("-", "")


def load_ecdsa_vectors(source) -> List[EcdsaVector]:
    """The secp256r1 tests of a Wycheproof ECDSA verification file (ecdsa_verify_schema / ecdsa_p1363_verify_schema):
    accepts a path, JSON text or a parsed dict.  Groups on other curves or of other types are left out.  A group
    with `"prehashed": true` carries the digest itself in `msg` (rows no message can produce, such as digest 0)."""
    if isinstance(source, dict):
        doc = source
    else:
        s = str(source)
        doc = json.loads(s) if s.lstrip().startswith("{") else json.load(open(s))
    out = []
    for g in doc.get("testGroups", []):
        enc = _ECDSA_GROUPS.get(g.get("type"))
        key = g.get("publicKey") or g.get("key") or {}
        if enc is None or key.get("curve") != "secp256r1":
            continue
        h = None if g.get("prehashed") else _hashlib_name(g["sha"])
        for t in g.get("tests", []):
            out.append(EcdsaVector(int(t.get("tcId", len(out) + 1)), t.get("comment", ""), t["msg"], t["sig"],
                                   t.get("result", "valid"), tuple(t.get("flags", ())), key["uncompressed"], h, enc))
    return out


def run_ecdsa_vectors(vectors: Sequence[EcdsaVector]):
    """All vectors of a suite in ONE call of the batch verifier.  A "valid" test passes when the signature verifies,
    an "invalid" one when it does not; "acceptable" tests (legacy encodings a verifier may accept or reject) always
    pass and are reported by the caller.  Returns (verified bool[n], passed bool[n])."""
    from .ecdsa import prepare, verify_digest

    n = len(vectors)
    rows = np.zeros((5, n, 32), dtype=np.uint8)
    parsed = np.zeros(n, dtype=bool)
    kinds = sorted({(v.hash or "", v.encoding) for v in vectors})
    for h, enc in kinds:
        idx = [i for i, v in enumerate(vectors) if (v.hash or "", v.encoding) == (h, enc)]
        part, ok = prepare([bytes.fromhex(vectors[i].msg) for i in idx], [bytes.fromhex(vectors[i].sig) for i in idx],
                           [bytes.fromhex(vectors[i].public_key) for i in idx], h or None, enc)
        for k in range(5):
            rows[k, idx] = part[k]
        parsed[idx] = ok
    verified = (verify_digest(*rows) & parsed) if n else parsed
    want = np.array([v.result == "valid" for v in vectors], dtype=bool)
    passed = (verified == want) | np.array([v.result == "acceptable" for v in vectors], dtype=bool)
    return verified, passed


# ---------------------------------------------------------------------------------------------
# Ed25519 suites through the batch verifier
# ---------------------------------------------------------------------------------------------
@dataclass
class EddsaVector:
    tc_id: int
    comment: str
    msg: str
    sig: str
    result: str
    flags: tuple
    public_key: str          # the 32-byte encoding A, hex


def load_eddsa_vectors(source) -> List[EddsaVector]:
    """The edwards25519 tests of a Wycheproof EdDSA verification file (eddsa_verify_schema): accepts a path, JSON
    text or a parsed dict.  The key is `publicKey.pk` (or `key.pk` in older files); groups on other curves (Ed448)
    or of other types are left out."""
    if isinstance(source, dict):
        doc = source
    else:
        s = str(source)
        doc = json.loads(s) if s.lstrip().startswith("{") else json.load(open(s))
    out = []
    for g in doc.get("testGroups", []):
        key = g.get("publicKey") or g.get("key") or {}
        if g.get("type") != "EddsaVerify" or key.get("curve") != "edwards25519":
            continue
        for t in g.get("tests", []):
            out.append(EddsaVector(int(t.get("tcId", len(out) + 1)), t.get("comment", ""), t["msg"], t["sig"],
                                   t.get("result", "valid"), tuple(t.get("flags", ())), key["pk"]))
    return out


def run_eddsa_vectors(vectors: Sequence[EddsaVector]):
    """All vectors of a suite in ONE call of the batch verifier.  A "valid" test passes when the signature verifies,
    an "invalid" one when it does not; "acceptable" tests always pass and are reported by the caller.  Returns
    (verified bool[n], passed bool[n])."""
    from .eddsa import verify

    verified = verify([bytes.fromhex(v.msg) for v in vectors], [bytes.fromhex(v.sig) for v in vectors],
                      [bytes.fromhex(v.public_key) for v in vectors])
    want = np.array([v.result == "valid" for v in vectors], dtype=bool)
    passed = (verified == want) | np.array([v.result == "acceptable" for v in vectors], dtype=bool)
    return verified, passed


def main(argv=None):
    """`python -m modarith_b200.wire FILE`: an ecdsa*/ed* file is converted as parse.py does (same
    lines on stdout); an x25519*/x448* file is run through the batch ladder and summarised."""
    import os
    import sys

    argv = sys.argv[1:] if argv is None else argv
    if len(argv) != 1:
        print("usage: python -m modarith_b200.wire <wycheproof file>", file=sys.stderr)
        return 2
    name = os.path.basename(argv[0]).lower()
    if name.startswith(("ecdsa", "ed")):
        sys.stdout.write(signature_lines(parse_signature_vectors(open(argv[0]).read(), name)))
        return 0
    curve = "X25519" if "25519" in name else ("X448" if "448" in name else None)
    if curve is None:
        print("cannot tell the curve from the file name", file=sys.stderr)
        return 1
    vecs = load_xdh_vectors(argv[0])
    _, passed = run_xdh_vectors(curve, vecs)
    for v, ok in zip(vecs, passed):
        if not ok:
            print("FAILED tcId %d (%s): %s" % (v.tc_id, v.result, v.comment))
    print("%s: %d tests, %d passed" % (curve, len(vecs), int(passed.sum())))
    return 0 if passed.all() else 1


if __name__ == "__main__":
    raise SystemExit(main())
