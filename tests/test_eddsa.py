"""Ed25519 verification without a GPU: the oracle against RFC 8032, OpenSSL and libsodium, the device code
(Eddsa::verify, Edwards::decode) on the host simulation over every fixture row and every decoding edge, the
reproducibility of the order field's header, the constant-time audit of k_eddsa_verify, and the host-side API."""
import ctypes
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import eddsa_oracle as O
from modarith_b200 import eddsa, wire
from modarith_b200 import lib as mlib

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
GOLDEN = os.path.join(ROOT, "tests", "golden", "eddsa_ed25519_sample.json")
FLAG = "NonCanonicalPublicKey"

crypto = pytest.importorskip("cryptography")
from cryptography.exceptions import InvalidSignature  # noqa: E402
from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey, Ed25519PublicKey  # noqa: E402
from cryptography.hazmat.primitives.serialization import Encoding, PublicFormat  # noqa: E402

RFC8032 = [  # section 7.1 TEST 1 and TEST 2: secret key, public key, message, signature
    ("9d61b19deffd5a60ba844af492ec2cc44449c5697b326919703bac031cae7f60",
     "d75a980182b10ab7d54bfed3c964073a0ee172f3daa62325af021a68f707511a", "",
     "e5564300c360ac729086e2cc806e828a84877f1eb8e5d974d873e065224901555fb8821590a33bacc61e39701cf9b46bd25bf5f0595bbe24655141438e7a100b"),
    ("4ccd089b28ff96da9db6c346ec114e0f5b8a319f35aba624da8cf6ed4fb8a6fb",
     "3d4017c3e843895a92b70aa74d1b7ebc9c982ccf2ec4968cc0cd55f12af4660c", "72",
     "92a009a9f0d4cab8720e820b5f642540a2b27b5416503f8fb3762223ebdb69da085ac1e43e15996e458f3613d0f11d8c387b2eaeb4302aeeb00d291612bb0c00"),
]

# the comparison table of the verification policy: row comment -> (this policy, OpenSSL, libsodium)
POLICY_TABLE = {
    "honest signature": (True, True, True),
    "S replaced by S + L": (False, False, False),
    "A = identity, R = enc([S]B)": (True, True, False),
    "A = identity as y = p + 1 (non-canonical)": (False, True, False),
    "A = (0, 1) with the sign bit set": (False, True, False),
    "A = aB + T8, k = 0 mod 8": (True, True, True),
    "A = aB + T8, k != 0 mod 8 (a cofactored verifier would accept)": (False, False, False),
}


def _openssl(msg, sig, pk):
    try:
        Ed25519PublicKey.from_public_bytes(pk).verify(sig, msg)
        return True
    except (InvalidSignature, ValueError):
        return False


def _raw(v):
    return bytes.fromhex(v.msg), bytes.fromhex(v.sig), bytes.fromhex(v.public_key)


@pytest.fixture(scope="module")
def vectors():
    return wire.load_eddsa_vectors(GOLDEN)


@pytest.fixture(scope="module")
def sim(tmp_path_factory):
    """g++ build of tests/hostsim/hostsim_eddsa.cpp: Eddsa::verify and Edwards::decode with the PTX blocks
    transcribed to C."""
    from modarith_b200.gen.cli import generate_all
    d = tmp_path_factory.mktemp("hostsim_eddsa")
    generate_all(verbose=False, outdir=str(d))           # fresh headers in a scratch directory, not in the source tree
    out = str(d / "libhostsim_eddsa.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-w", "-I", str(d),
                           "-I", os.path.join(ROOT, "modarith_b200", "csrc"),
                           "-o", out, os.path.join(ROOT, "tests", "hostsim", "hostsim_eddsa.cpp")])
    lib = ctypes.CDLL(out)
    lib.sim_ED25519_eddsa_verify.restype = ctypes.c_int
    lib.sim_ED25519_decode.restype = ctypes.c_int
    return lib


def test_oracle_reproduces_rfc8032_vectors():
    for sk, pk, msg, sig in RFC8032:
        sk, pk, msg, sig = (bytes.fromhex(x) for x in (sk, pk, msg, sig))
        assert O.public_key(sk) == pk and O.sign(sk, msg) == sig
        assert O.verify(msg, sig, pk)
        k = Ed25519PrivateKey.from_private_bytes(sk)
        assert k.public_key().public_bytes(Encoding.Raw, PublicFormat.Raw) == pk and k.sign(msg) == sig


def test_fixture_covers_the_policy_table(vectors):
    by = {}
    for v in vectors:
        by.setdefault(v.comment, set()).add(v.result)
    for comment, (ours, _, _) in POLICY_TABLE.items():
        assert by[comment] == {"valid" if ours else "invalid"}, comment
    for c in ("RFC 8032 7.1 TEST 1", "RFC 8032 7.1 TEST 2", "S = L - 1", "S = L", "S = 2^255 - 1", "S = 2^256 - 1",
              "S = 2^255 (only bit 255 set)", "key y = p - 1 with the sign bit (x = 0)", "R with its sign bit flipped",
              "non-canonical R: the identity as y = p + 1", "R of order 2, S = 0, A of order 2", "empty message",
              "1 KiB message", "wrong message", "wrong key", "signature of 63 bytes", "signature of 65 bytes",
              "key of 31 bytes"):
        assert c in by, c
    assert by["S = L - 1"] == by["R of order 2, S = 0, A of order 2"] == {"valid"}
    noncanon = [v for v in vectors if v.comment.startswith("non-canonical key")]
    ys = {int(v.comment.split()[4]) for v in noncanon}
    assert ys == {y for y in range(19) if O.recover_x(y, 0) is not None}
    assert len(noncanon) == 2 * len(ys)
    assert any(v.comment.endswith("has no square root") for v in vectors)


def test_oracle_agrees_with_openssl_on_the_fixture(vectors):
    flagged = 0
    for v in vectors:
        msg, sig, pk = _raw(v)
        ours = O.verify(msg, sig, pk)
        assert ours == (v.result == "valid"), (v.tc_id, v.comment)
        if FLAG in v.flags:                              # OpenSSL decodes these keys leniently and accepts
            assert _openssl(msg, sig, pk) and not ours, (v.tc_id, v.comment)
            flagged += 1
        else:
            assert _openssl(msg, sig, pk) == ours, (v.tc_id, v.comment)
    kinds = {v.comment for v in vectors if FLAG in v.flags}
    assert flagged >= 4 and "A = identity as y = p + 1 (non-canonical)" in kinds and "A = (0, 1) with the sign bit set" in kinds


def test_policy_table_openssl_and_libsodium_columns(vectors):
    nacl = pytest.importorskip("nacl.signing")
    from nacl.exceptions import BadSignatureError

    def sodium(msg, sig, pk):
        try:
            nacl.VerifyKey(pk).verify(msg, sig)
            return True
        except (BadSignatureError, ValueError):
            return False

    seen = set()
    for v in vectors:
        if v.comment not in POLICY_TABLE:
            continue
        ours, openssl, libsodium = POLICY_TABLE[v.comment]
        msg, sig, pk = _raw(v)
        assert (O.verify(msg, sig, pk), _openssl(msg, sig, pk), sodium(msg, sig, pk)) == (ours, openssl, libsodium), v.comment
        seen.add(v.comment)
    assert seen == set(POLICY_TABLE)


def test_oracle_agrees_with_openssl_on_random_signatures():
    rng = random.Random(2000)
    keys = [Ed25519PrivateKey.from_private_bytes(rng.randbytes(32)) for _ in range(16)]
    pubs = [k.public_key().public_bytes(Encoding.Raw, PublicFormat.Raw) for k in keys]
    mutated_valid = 0
    for i in range(2000):
        msg = rng.randbytes(rng.randrange(0, 64))
        sig, pk = keys[i % 16].sign(msg), pubs[i % 16]
        assert O.verify(msg, sig, pk) and _openssl(msg, sig, pk), i
        # one single-bit mutation of the message, the signature or the key
        blob = bytearray(msg + sig + pk)
        bit = rng.randrange(8 * len(blob))
        blob[bit >> 3] ^= 1 << (bit & 7)
        m2, s2, k2 = bytes(blob[:len(msg)]), bytes(blob[len(msg):len(msg) + 64]), bytes(blob[len(msg) + 64:])
        want = _openssl(m2, s2, k2)
        assert O.verify(m2, s2, k2) == want, (i, bit)
        mutated_valid += want
    assert mutated_valid == 0


def _sim_verify(sim, msg, sig, pk):
    rows, parsed = eddsa.prepare([msg], [sig], [pk])
    return bool(sim.sim_ED25519_eddsa_verify(*(r[0].tobytes() for r in rows))) and bool(parsed[0])


def test_hostsim_verifies_every_fixture_row(sim, vectors):
    for v in vectors:
        assert _sim_verify(sim, *_raw(v)) == (v.result == "valid"), (v.tc_id, v.comment)


def test_hostsim_agrees_with_the_oracle_on_mutations(sim):
    rng = random.Random(8032)
    for i in range(40):
        seed = rng.randbytes(32)
        msg = rng.randbytes(rng.randrange(0, 40))
        sig, pk = O.sign(seed, msg), O.public_key(seed)
        assert _sim_verify(sim, msg, sig, pk)
        s = bytearray(sig)
        s[rng.randrange(64)] ^= 1 << rng.randrange(8)
        assert _sim_verify(sim, msg, bytes(s), pk) == O.verify(msg, bytes(s), pk), i


def _sim_decode(sim, enc):
    x, y = ctypes.create_string_buffer(32), ctypes.create_string_buffer(32)
    ok = sim.sim_ED25519_decode(enc, x, y)
    return ok, (int.from_bytes(x.raw, "little"), int.from_bytes(y.raw, "little"))


def test_hostsim_decode_edges_match_the_oracle(sim):
    rng = random.Random(5113)
    nonsquares = [y for y in range(2, 200) if O.recover_x(y, 0) is None][:8]
    ys = [O.P + y for y in range(19)] + [O.P - 1, O.P - 2, 0, 1] + nonsquares + [rng.randrange(O.P) for _ in range(64)]
    ys += [(1 << 255) - 1, (1 << 255) - 2]
    rejected = 0
    for y in ys:
        for sign in (0, 1):
            enc = (y | (sign << 255)).to_bytes(32, "little")
            ok, pt = _sim_decode(sim, enc)
            want = O.decode(enc)
            assert ok == (want is not None), (hex(y), sign)
            assert pt == (want if want is not None else O.IDENTITY), (hex(y), sign)
            rejected += want is None
    assert rejected > 2 * 19


def test_hostsim_reduces_the_digest_mod_L(sim):
    rng = random.Random(512)
    vals = [0, O.L - 1, O.L, (1 << 256) - 1, 1 << 256, O.L << 256, (1 << 512) - 1] + [rng.randrange(1 << 512) for _ in range(50)]
    for v in vals:
        k = ctypes.create_string_buffer(32)
        sim.sim_ED25519_reduce512(v.to_bytes(64, "little"), k)
        assert int.from_bytes(k.raw, "little") == v % O.L, hex(v)


def test_order_field_header_is_the_generators_output(tmp_path):
    """The header the build compiles (generated into the build directory, not committed) is what the generator prints,
    the same on every run, and the only copy the X25519 unit can include."""
    from modarith_b200.build import OBJDIR, build
    from modarith_b200.gen.cli import generate
    from modarith_b200.gen.plan import MontgomeryFull, make_plan
    from modarith_b200.primes import ALL_PRIMES, ORDER_PRIMES
    P = ORDER_PRIMES["ED25519ORDER"]
    assert P.p == O.L and isinstance(make_plan(P), MontgomeryFull) and make_plan(P).L == 8
    build(verbose=False)
    a = open(generate(P, str(tmp_path / "a" / "field_ED25519ORDER.cuh"), verbose=False)).read()
    b = open(generate(P, str(tmp_path / "b" / "field_ED25519ORDER.cuh"), verbose=False)).read()
    assert a == b == open(os.path.join(OBJDIR, "gen", "field_ED25519ORDER.cuh")).read()
    assert "struct F_ED25519ORDER" in a and "MontgomeryFull" in a
    assert not os.path.exists(os.path.join(ROOT, "modarith_b200", "csrc", "gen", "field_ED25519ORDER.cuh"))
    assert "ED25519ORDER" not in ALL_PRIMES and "ED25519ORDER" not in mlib.PRIMES


def test_k_eddsa_verify_audits_clean():
    from modarith_b200.build import build, OBJDIR
    build(verbose=False)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ct_audit
    found = 0
    for name, ins in ct_audit.parse(os.path.join(OBJDIR, "mab_capi_X25519.o"), "k_eddsa_verify"):
        flags, _, _ = ct_audit.analyse(name, ins)
        assert flags == [], [(w, d["text"]) for w, d in flags[:10]]
        found += 1
    assert found == 1
    assert ("mab_capi_X25519.o", "k_eddsa") in ct_audit.DEFAULT


def test_no_order_field_entry_points_are_exported():
    from modarith_b200.build import build
    so = build(verbose=False)
    out = subprocess.run(["nm", "-D", "--defined-only", so], stdout=subprocess.PIPE, text=True)
    if out.returncode != 0:
        pytest.skip("nm not available")
    assert "mab_ED25519_eddsa_verify" in out.stdout and "ED25519ORDER" not in out.stdout


def test_argument_errors_need_no_gpu():
    with pytest.raises(ValueError):
        eddsa.verify([b"m", b"n"], [bytes(64)], [bytes(32)])
    with pytest.raises(ValueError):
        eddsa.prepare([b"m"], [bytes(64), bytes(64)], [bytes(32)])
    assert eddsa.verify([], [], []).shape == (0,)
    h, s, k = np.zeros((2, 64), np.uint8), np.zeros((2, 64), np.uint8), np.zeros((2, 32), np.uint8)
    for bad in ((h[:, :32], s, k), (h, s[:, :63], k), (h, s, np.zeros((2, 64), np.uint8)), (h, s, k[:1]),
                (h.astype(np.int16), s, k), (h[None], s, k), (h[:, ::2], s, k)):
        with pytest.raises(ValueError):
            eddsa.verify_digest(*bad)
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(mlib.MabError):
            eddsa.verify_digest(h, s, k)                  # no CPU fallback


def test_prepare_zeroes_unparsed_rows_and_verify_masks_them(monkeypatch):
    rng = random.Random(4)
    seed = rng.randbytes(32)
    msg = b"abc"
    sig, pk = O.sign(seed, msg), O.public_key(seed)
    (h, s, k), parsed = eddsa.prepare([msg] * 4, [sig, sig[:63], sig + b"\x00", sig], [pk, pk, pk, pk[:31]])
    assert list(parsed) == [True, False, False, False]
    assert h[0].tobytes() == O.digest(sig[:32], pk, msg) and s[0].tobytes() == sig and k[0].tobytes() == pk
    assert not h[1:].any() and not s[1:].any() and not k[1:].any()
    # the kernel is not asked to reject zero rows: whatever it says about them, verify() reports parsed rows only
    monkeypatch.setattr(eddsa, "verify_digest", lambda *rows: np.ones(rows[0].shape[0], dtype=bool))
    assert list(eddsa.verify([msg] * 4, [sig, sig[:63], sig + b"\x00", sig], [pk, pk, pk, pk[:31]])) == list(parsed)


def test_wycheproof_loader_takes_either_key_field_and_skips_other_curves():
    doc = json.load(open(GOLDEN))
    g = doc["testGroups"][0]
    old = dict(g, key=g["publicKey"])
    del old["publicKey"]
    ed448 = dict(g, publicKey=dict(g["publicKey"], curve="edwards448"))
    other = dict(g, type="XdhComp")
    vs = wire.load_eddsa_vectors({"testGroups": [g, old, ed448, other]})
    assert len(vs) == 2 * len(g["tests"]) and {v.public_key for v in vs} == {g["publicKey"]["pk"]}
    assert len(wire.load_eddsa_vectors(GOLDEN)) == doc["numberOfTests"]
