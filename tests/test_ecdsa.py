"""ECDSA P-256 verification without a GPU: the oracle against OpenSSL, the strict DER parser against cryptography's,
the device code (Ecdsa::verify) on the host simulation over every fixture row, the constant-time audit of
k_ecdsa_verify, the C ABI of include/modarith_b200_sig.h, and the argument checks."""
import ctypes
import hashlib
import json
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest

import ecdsa_oracle as O
from modarith_b200 import ecdsa, wire
from modarith_b200 import lib as mlib

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
GOLDEN = [os.path.join(ROOT, "tests", "golden", f) for f in ("ecdsa_secp256r1_sha256_sample.json",
                                                             "ecdsa_secp256r1_sha256_p1363_sample.json")]

crypto = pytest.importorskip("cryptography")
from cryptography.exceptions import InvalidSignature  # noqa: E402
from cryptography.hazmat.primitives import hashes  # noqa: E402
from cryptography.hazmat.primitives.asymmetric import ec, utils  # noqa: E402


def _openssl(v):
    try:
        pk = ec.EllipticCurvePublicKey.from_encoded_point(ec.SECP256R1(), bytes.fromhex(v.public_key))
    except ValueError:
        return False
    sig = bytes.fromhex(v.sig)
    if v.encoding == "p1363":
        if len(sig) != 64:
            return False
        sig = utils.encode_dss_signature(int.from_bytes(sig[:32], "big"), int.from_bytes(sig[32:], "big"))
    try:
        pk.verify(sig, bytes.fromhex(v.msg), ec.ECDSA(utils.Prehashed(hashes.SHA256()) if v.hash is None else hashes.SHA256()))
        return True
    except InvalidSignature:
        return False


def _oracle(v):
    key = bytes.fromhex(v.public_key)
    sig = bytes.fromhex(v.sig)
    try:
        r, s = utils.decode_dss_signature(sig) if v.encoding == "der" else ecdsa.decode_p1363(sig)
    except ValueError:
        return False
    d = bytes.fromhex(v.msg) if v.hash is None else hashlib.new(v.hash, bytes.fromhex(v.msg)).digest()
    q = (int.from_bytes(key[1:33], "big"), int.from_bytes(key[33:], "big"))
    return O.verify(O.bits2int(d), r, s, q)


@pytest.fixture(scope="module")
def sim(tmp_path_factory):
    """g++ build of tests/hostsim/hostsim_ecdsa.cpp: Ecdsa::verify with the PTX blocks transcribed to C."""
    from modarith_b200.gen.cli import generate_all
    d = tmp_path_factory.mktemp("hostsim_ecdsa")
    generate_all(verbose=False, outdir=str(d))           # fresh headers in a scratch directory, not in the source tree
    out = str(d / "libhostsim_ecdsa.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-w", "-I", str(d),
                           "-I", os.path.join(ROOT, "modarith_b200", "csrc"),
                           "-o", out, os.path.join(ROOT, "tests", "hostsim", "hostsim_ecdsa.cpp")])
    lib = ctypes.CDLL(out)
    lib.sim_NIST256_ecdsa_verify.restype = ctypes.c_int
    return lib


@pytest.fixture(scope="module")
def vectors():
    return [wire.load_ecdsa_vectors(p) for p in GOLDEN]


def test_fixture_covers_the_edge_cases(vectors):
    der, p1363 = vectors
    comments = {v.comment for v in der}
    for c in ("r = 0", "s = n", "r = 2^256 - 1", "r = s = 1", "digest 0", "digest n", "digest 2^256 - 1",
              "h = -r d: u1 G + u2 Q = O", "x(R) in [n, p): r = x(R) - n", "x(R) in [n, p): r = x(R) unreduced",
              "r = p - n - 1", "r = p - n", "public key off the curve", "key coordinate x + p", "Q = G", "Q = -G",
              "DER: indefinite length", "DER: missing s", "DER: negative INTEGER"):
        assert c in comments, c
    by = {v.comment: v.result for v in der}
    assert by["x(R) in [n, p): r = x(R) - n"] == "valid" and by["x(R) in [n, p): r = x(R) unreduced"] == "invalid"
    assert {v.encoding for v in der} == {"der"} and {v.encoding for v in p1363} == {"p1363"}
    assert sum(v.result == "valid" for v in p1363) == sum(v.result == "valid" for v in der) == 20


def test_oracle_agrees_with_openssl_on_the_fixture(vectors):
    for vs in vectors:
        for v in vs:
            assert _oracle(v) == _openssl(v) == (v.result == "valid"), (v.tc_id, v.comment)


def test_oracle_agrees_with_openssl_on_random_signatures():
    rng = random.Random(2000)
    keys = [ec.derive_private_key(rng.randrange(1, O.N), ec.SECP256R1()) for _ in range(16)]
    algo = ec.ECDSA(hashes.SHA256())
    for i in range(2000):
        k = keys[i % 16]
        msg = rng.randbytes(rng.randrange(0, 64))
        r, s = utils.decode_dss_signature(k.sign(msg, algo))
        pn = k.public_key().public_numbers()
        kind = i % 4                                   # 0 as signed, 1 s -> n - s, 2 other message, 3 other key
        if kind == 1:
            s = O.N - s
        if kind == 2:
            msg += b"\x00"
        if kind == 3:
            pn = keys[(i + 1) % 16].public_key().public_numbers()
        try:
            ec.EllipticCurvePublicNumbers(pn.x, pn.y, ec.SECP256R1()).public_key().verify(
                utils.encode_dss_signature(r, s), msg, algo)
            want = True
        except InvalidSignature:
            want = False
        assert want == (kind < 2)
        assert O.verify(O.bits2int(hashlib.sha256(msg).digest()), r, s, (pn.x, pn.y)) == want, i


def _decode_both(sig):
    try:
        a = utils.decode_dss_signature(sig)
    except ValueError:
        a = None
    try:
        b = ecdsa.decode_der(sig)
    except ValueError:
        b = None
    return a, b


def test_der_parser_accepts_exactly_what_cryptography_accepts(vectors):
    der = vectors[0]
    sigs = [bytes.fromhex(v.sig) for v in der]
    for sig in sigs:
        a, b = _decode_both(sig)
        assert a == b, sig.hex()
    # every single-byte change, truncation and extension of one well-formed signature
    good = next(bytes.fromhex(v.sig) for v in der if v.result == "valid")
    rng = random.Random(7)
    cands = [good[:k] for k in range(len(good))] + [good + bytes([x]) for x in (0, 1, 0x30)]
    for k in range(len(good)):
        for x in (0x00, 0x01, 0x7f, 0x80, 0x81, 0xff, good[k] ^ 1, rng.randrange(256)):
            cands.append(good[:k] + bytes([x]) + good[k + 1:])
    accepted = 0
    for sig in cands:
        a, b = _decode_both(sig)
        assert a == b, sig.hex()
        accepted += a is not None
    assert 0 < accepted < len(cands)


def _sim_rows(sim, vs):
    fn = sim.sim_NIST256_ecdsa_verify
    out = []
    for h, enc in sorted({(v.hash or "", v.encoding) for v in vs}):
        part = [v for v in vs if (v.hash or "", v.encoding) == (h, enc)]
        rows, parsed = ecdsa.prepare([bytes.fromhex(v.msg) for v in part], [bytes.fromhex(v.sig) for v in part],
                                     [bytes.fromhex(v.public_key) for v in part], h or None, enc)
        for i, v in enumerate(part):
            ok = fn(*(rows[k][i].tobytes() for k in range(5)))
            out.append((v, bool(ok) and bool(parsed[i])))
    return out


def test_hostsim_verifies_every_fixture_row(sim, vectors):
    for vs in vectors:
        got = _sim_rows(sim, vs)
        assert len(got) == len(vs)
        for v, ok in got:
            assert ok == (v.result == "valid"), (v.tc_id, v.comment)


def test_hostsim_rejects_what_the_host_lets_through(sim):
    """Rows the parser passes on unchanged: the device code alone must reject them."""
    fn = sim.sim_NIST256_ecdsa_verify
    b = lambda v: (v % (1 << 256)).to_bytes(32, "big")
    rng = random.Random(11)
    d = rng.randrange(1, O.N)
    Q = O.public_key(d)
    h = rng.randrange(1 << 200)
    r, s = O.sign(d, h, rng.randrange(1, O.N))
    assert fn(b(h), b(r), b(s), b(Q[0]), b(Q[1])) == 1
    assert fn(b(h + O.N), b(r), b(s), b(Q[0]), b(Q[1])) == 1                         # h >= n reduces
    for rr, ss in ((0, s), (r, 0), (O.N, s), (r, O.N), (r + O.N, s), (r, s + O.N), (0, 0)):
        if rr < 1 << 256 and ss < 1 << 256:
            assert fn(b(h), b(rr), b(ss), b(Q[0]), b(Q[1])) == 0, (rr, ss)
    if Q[0] + O.P < 1 << 256:
        assert fn(b(h), b(r), b(s), b(Q[0] + O.P), b(Q[1])) == 0
    if Q[1] + O.P < 1 << 256:
        assert fn(b(h), b(r), b(s), b(Q[0]), b(Q[1] + O.P)) == 0
    assert fn(b(h), b(r), b(s), b(0), b(0)) == 0


def test_k_ecdsa_verify_audits_clean():
    from modarith_b200.build import build, OBJDIR
    build(verbose=False)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ct_audit
    found = 0
    for name, ins in ct_audit.parse(os.path.join(OBJDIR, "mab_capi_NIST256.o"), "k_ecdsa_verify"):
        flags, _, _ = ct_audit.analyse(name, ins)
        assert flags == [], [(w, d["text"]) for w, d in flags[:10]]
        found += 1
    assert found == 1
    assert ("mab_capi_NIST256.o", "k_ecdsa") in ct_audit.DEFAULT


def test_signature_header_symbols_are_exported(tmp_path):
    from modarith_b200.build import build
    so = build(verbose=False)
    h = open(os.path.join(ROOT, "include", "modarith_b200_sig.h")).read()
    assert set(re.findall(r"\b(mab_[A-Za-z0-9_]+)\s*\(", h)) == set(mlib.signature_symbols())
    assert not set(mlib.signature_symbols()) & set(mlib.exported_symbols())
    dll = ctypes.CDLL(so)
    for s in mlib.signature_symbols():
        assert hasattr(dll, s), s
    import shutil
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    src = tmp_path / "consumer.c"
    src.write_text(
        '#include <stdio.h>\n#include "modarith_b200_sig.h"\n'
        "int main(void) {\n"
        "  int (*v)(const char *, const char *, const char *, const char *, const char *, unsigned char *, size_t, void *) =\n"
        "      mab_NIST256_ecdsa_verify;\n"
        "  int (*mul2)(const char *, const char *, const char *, const char *, const char *, const char *, char *, char *, size_t, void *) = mab_NIST256_ecnmul2;\n"
        "  if (!v || !mul2) return 2;\n"
        '  printf("%s\\n", mab_version());\n'
        "  return v(0, 0, 0, 0, 0, 0, 0, 0);                 /* n = 0: nothing to do, no device needed */\n"
        "}\n")
    exe = tmp_path / "consumer"
    libdir = os.path.dirname(so)
    subprocess.check_call(["gcc", "-std=c11", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src),
                           "-L", libdir, "-lmodarith_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    out = subprocess.run([str(exe)], stdout=subprocess.PIPE, text=True)
    assert out.returncode == 0 and out.stdout.startswith("modarith_b200")


def test_argument_errors_need_no_gpu():
    key = b"\x04" + bytes(64)
    with pytest.raises(ValueError):
        ecdsa.verify([b"m"], [b"s"], [key], encoding="ber")
    with pytest.raises(ValueError):
        ecdsa.verify([b"m", b"n"], [b"s"], [key])
    with pytest.raises(ValueError):
        ecdsa.verify([b"m"], [b"s"], [key], hash="no-such-hash")
    assert ecdsa.verify([], [], []).shape == (0,)
    for bad in (b"", b"\x04" + bytes(63), b"\x02" + bytes(64)):
        with pytest.raises(ValueError):
            ecdsa.decode_public_key(bad)
    with pytest.raises(ValueError):
        ecdsa.decode_p1363(bytes(63))
    import torch
    if not torch.cuda.is_available():
        a = np.zeros((2, 32), dtype=np.uint8)
        with pytest.raises(mlib.MabError):
            ecdsa.verify_digest(a, a, a, a, a)             # no CPU fallback


def test_prepare_rows():
    """bits2int keeps the leftmost 256 bits (SHA-384, SHA-512); unparsable rows are zeros and not parsed."""
    rng = random.Random(3)
    k = ec.derive_private_key(rng.randrange(1, O.N), ec.SECP256R1())
    from cryptography.hazmat.primitives.serialization import Encoding, PublicFormat
    key = k.public_key().public_bytes(Encoding.X962, PublicFormat.UncompressedPoint)
    msg = b"abc"
    for name, algo in (("sha256", hashes.SHA256()), ("sha384", hashes.SHA384()), ("sha512", hashes.SHA512())):
        sig = k.sign(msg, ec.ECDSA(algo))
        rows, parsed = ecdsa.prepare([msg, msg], [sig, sig + b"\x00"], [key, key], name, "der")
        assert list(parsed) == [True, False] and not rows[0][1].any() and not rows[1][1].any()
        d = hashlib.new(name, msg).digest()
        assert rows[0][0].tobytes() == d[:32]
        r, s = utils.decode_dss_signature(sig)
        assert (rows[1][0].tobytes(), rows[2][0].tobytes()) == (r.to_bytes(32, "big"), s.to_bytes(32, "big"))
        assert O.verify(O.bits2int(d), r, s, O.public_key(k.private_numbers().private_value))


def test_wire_still_prints_parse_lines_for_ecdsa_files():
    text = open(GOLDEN[0]).read()
    recs = wire.parse_signature_vectors(text, "ecdsa_secp256r1_sha256_sample.json")
    doc = json.load(open(GOLDEN[0]))
    assert len(recs) == doc["numberOfTests"]
    assert [r.result for r in recs] == [t["result"] for g in doc["testGroups"] for t in g["tests"]]
