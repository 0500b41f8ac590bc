"""The add-on library of a modulus outside the built-in five (python -m modarith_b200.build --prime NIST384) on the
GPU: the same entry points, checked byte-for-byte against the reference's own generated C for that modulus
(`monty.py 64 NIST384`, oracle/_ref/libref_NIST384.so) and against the value-level oracle."""
import os
import random
import sys

import numpy as np
import pytest
import torch

import util
from field_oracle import FieldOracle
from oracle_primes import OraclePrime

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
P384 = 2**384 - 2**128 - 2**96 + 2**32 - 1            # monty.py named table, "NIST384"
# add-on moduli: 2^414 - 17 (13 limbs, two spare bits) and
# 2^521 - 1 (17 limbs, 23 spare bits) take the bit-level pseudo-Mersenne plan (pseudo.py named table)
# 5*2^248 - 1 (monty.py named table "ED248") and NIST384 itself are p = -1 (mod 2^(32z)), z = 7 and 1: the
# Montgomery-friendly plan
ADDONS = {"NIST384": P384, "C41417": 2**414 - 17, "NIST521": 2**521 - 1, "ED248": 5 * 2**248 - 1}


@pytest.fixture(scope="module")
def F():
    from modarith_b200 import Field, lib as mlib
    if not os.path.exists(mlib.extra_lib_path("NIST384")):
        pytest.fail("libmodarith_b200_NIST384.so is missing: __graft_entry__.build() builds it")
    return Field("NIST384")


def _bytes(t):
    return t.cpu().numpy()


def _oracle_field_batch(name, op, a, b=None):
    """The value-level oracle row by row, shaped like util.ref_field_batch's (outputs, status)."""
    O = FieldOracle(OraclePrime(name, ADDONS[name]))
    nb = a.shape[1]
    out, st = np.zeros_like(a), np.zeros(a.shape[0], dtype=np.int32)
    for i in range(a.shape[0]):
        bv = None if b is None else int.from_bytes(b[i].tobytes(), "big")
        v, st[i] = util.oracle_field_op(O, op, int.from_bytes(a[i].tobytes(), "big"), bv)
        out[i] = np.frombuffer(v.to_bytes(nb, "big"), dtype=np.uint8)
    return out, st


@pytest.mark.parametrize("name", list(ADDONS))
def test_field_ops_vs_reference_build(name):
    """Six operations on 4096 elements against the reference's own generated C for the modulus (oracle/_ref).  Where
    that build is absent: the corner rows and a fixed sample of 512 others against the value-level oracle, which no
    stored reference vector covers for these moduli, so every nonzero inverse and every square root of a square is
    also checked by its defining identity."""
    import ctypes
    from modarith_b200 import Field, lib as mlib
    if not os.path.exists(mlib.extra_lib_path(name)):
        pytest.fail("libmodarith_b200_%s.so is missing: __graft_entry__.build() builds it" % name)
    path = os.path.join(ROOT, "oracle", "_ref", "libref_%s.so" % name)
    ref = ctypes.CDLL(path) if os.path.exists(path) else None
    F = Field(name)
    p = ADDONS[name]
    nb, n = F.Nbytes, 1 << 12
    assert nb == (p.bit_length() + 7) // 8 and F.Nlimbs == (p.bit_length() + 31) // 32
    a, b = util.random_bytes(384, n, nb), util.random_bytes(385, n, nb)
    top = 1 << p.bit_length()
    # the reference's modimp takes values below 2p (SURVEY.md 8b): keep the random rows inside the field's bit length
    spare = 8 * nb - p.bit_length()
    if spare:
        a[:, 0] &= 0xFF >> spare
        b[:, 0] &= 0xFF >> spare
    for i, v in enumerate([p - 1, p, p + 1, top - 1, 0, 1, p - 2, (p + top) // 2]):
        a[i] = np.frombuffer(v.to_bytes(nb, "big"), dtype=np.uint8)
    x, st = F.modimp(torch.from_numpy(a).cuda())
    y, _ = F.modimp(torch.from_numpy(b).cuda())
    r = F.alloc(n)
    rows = np.arange(n) if ref is not None else util.sample_rows(n, 512, head=8)
    for op in ("mul", "sqr", "inv", "sqrt", "add", "sub"):
        bb = b[rows] if op in ("mul", "add", "sub") else None
        want, wst = util.ref_field_batch(ref, op, a, bb) if ref is not None else _oracle_field_batch(name, op, a[rows], bb)
        if op == "mul": F.modmul(x, y, r)
        if op == "sqr": F.modsqr(x, r)
        if op == "inv": F.modinv(x, None, r)
        if op == "sqrt": F.modsqrt(x, None, r)
        if op == "add": F.modadd(x, y, r)
        if op == "sub": F.modsub(x, y, r)
        got = _bytes(F.modexp(r))[rows]
        assert np.array_equal(got, want), (name, op)
        assert np.array_equal(st.cpu().numpy()[rows], wst), (name, op)
        if ref is None and op in ("inv", "sqrt"):
            for i, g in zip(rows, got):
                av, gv = int.from_bytes(a[i].tobytes(), "big") % p, int.from_bytes(g.tobytes(), "big")
                if op == "inv" and av:
                    assert av * gv % p == 1, (name, i)
                if op == "sqrt" and pow(av, (p - 1) // 2, p) in (0, 1):
                    assert gv * gv % p == av, (name, i)


@pytest.mark.parametrize("name", ["C41417", "NIST521"])
def test_bit_level_pseudo_mersenne_plan_api_vs_oracle(name):
    """The rest of the API on the bit-level plan (values stored below 2^n + 2^32, raw imports up to 2^(32L))."""
    from modarith_b200 import Field
    p = ADDONS[name]
    F = Field(name)
    O = FieldOracle(OraclePrime(name, p))
    rng = random.Random(521)
    xs = [0, 1, 2, p - 1, p - 2, (p - 1) // 2] + [rng.randrange(p) for _ in range(300)]
    ys = [p - 1, 0, 1, 2, p - 1, 3] + [rng.randrange(p) for _ in range(300)]
    x, y = F.from_ints(xs), F.from_ints(ys)
    r = F.alloc(len(xs))
    F.modneg(x, r); assert F.to_ints(r) == [O.modneg(a) for a in xs]
    F.modmli(x, 121665, r); assert F.to_ints(r) == [O.modmli(a, 121665) for a in xs]
    F.modmli(x, (1 << 31) - 1, r); assert F.to_ints(r) == [O.modmli(a, (1 << 31) - 1) for a in xs]
    F.modcpy(x, r); F.modhaf(r); assert F.to_ints(r) == [O.modhaf(a) for a in xs]
    F.modcpy(x, r); F.modnsqr(r, 5); assert F.to_ints(r) == [O.modnsqr(a, 5) for a in xs]
    F.modpro(x, r); assert F.to_ints(r) == [O.modpro(a) for a in xs]
    assert F.modqr(None, x).cpu().tolist() == [O.modqr(None, a) for a in xs]
    assert F.modis0(x).cpu().tolist() == [int(a == 0) for a in xs]
    assert F.modis1(x).cpu().tolist() == [int(a == 1) for a in xs]
    assert F.modcmp(x, y).cpu().tolist() == [int(a == b) for a, b in zip(xs, ys)]
    assert F.modsign(x).cpu().tolist() == [a & 1 for a in xs]
    # a long chain keeps the representation inside its bound: ((x*y + x - y)^2 * 7 - x)^-1 ...
    code = [("mul", 2, 0, 1), ("add", 2, 2, 0), ("sub", 2, 2, 1), ("sqr", 2, 2, 0), ("mli", 2, 2, 0, 7), ("sub", 2, 2, 0),
            ("neg", 3, 2, 0), ("add", 3, 3, 3), ("mul", 3, 3, 2), ("inv", 4, 3, 0)]
    def ref(a, b):
        t = ((a * b + a - b) ** 2 * 7 - a) % p
        u = (-t * 2 * t) % p
        return pow(u, -1, p) if u else 0
    want = [ref(a, b) for a, b in zip(xs, ys)]
    for jit in (False, True):
        (res,) = F.modprog(code, [x, y], [4], jit=jit)
        assert F.to_ints(res) == want, (name, jit)
    # raw words up to 2^(32L) through nres (modimp of words): canonical value and the "< p" flag
    L = F.Nlimbs
    topw = 1 << (32 * L)
    raw = [topw - 1, topw - 2, p, p + 1, 2 * p, 3 * p + 5, topw >> 1, 0, p - 1] + [rng.randrange(topw) for _ in range(100)]
    planes = np.zeros((L, len(raw)), dtype=np.uint32)
    for i, v in enumerate(raw):
        for j in range(L):
            planes[j, i] = (v >> (32 * j)) & 0xFFFFFFFF
    t = torch.from_numpy(planes.view(np.int32)).cuda()
    flags = F.modfsb(t).cpu().tolist()
    assert flags == [int(v < p) for v in raw]
    got = t.cpu().numpy().view(np.uint32).astype(object)
    assert [sum(int(got[j, i]) << (32 * j) for j in range(L)) for i in range(len(raw))] == [v % p for v in raw]


def test_api_vs_oracle_and_programs(F):
    O = FieldOracle(OraclePrime("NIST384", P384))
    p = O.p
    rng = random.Random(384)
    xs = [0, 1, p - 1, p - 2] + [rng.randrange(p) for _ in range(200)]
    ys = [p - 1, 0, 1, 2] + [rng.randrange(p) for _ in range(200)]
    x, y = F.from_ints(xs), F.from_ints(ys)
    r = F.alloc(len(xs))
    F.modmul(x, y, r); assert F.to_ints(r) == [O.modmul(a, b) for a, b in zip(xs, ys)]
    F.modsub(x, y, r); assert F.to_ints(r) == [O.modsub(a, b) for a, b in zip(xs, ys)]
    F.modmli(x, 39081, r); assert F.to_ints(r) == [O.modmli(a, 39081) for a in xs]
    F.modcpy(x, r); F.modhaf(r); assert F.to_ints(r) == [O.modhaf(a) for a in xs]
    F.modpro(x, r); assert F.to_ints(r) == [O.modpro(a) for a in xs]
    assert F.modqr(None, x).cpu().tolist() == [O.modqr(None, a) for a in xs]
    code = [("mul", 2, 0, 1), ("add", 3, 2, 0), ("sqr", 3, 3, 0), ("sub", 4, 3, 1), ("mli", 5, 4, 0, 7), ("neg", 6, 5, 0)]
    want = [(-(7 * ((a * b + a) ** 2 - b))) % p for a, b in zip(xs, ys)]
    for jit in (False, True):
        (res,) = F.modprog(code, [x, y], [6], jit=jit)
        assert F.to_ints(res) == want, jit


# ---- a user-defined Montgomery curve: the add-on library's ladder ------------------------------------------------------
M383_P = 2**383 - 187


def _expected_m383(name, k, u, rows):
    """Rows `rows` of the ladder's expected output: the reference's rfc7748.c with the curve's constants
    (oracle/_ref/libref_<name>.so) on the whole batch where that build exists, otherwise the value-level oracle on
    those rows alone.  No stored reference vector covers this curve; where the build exists,
    tests/test_extra_modulus.py pins the oracle to it.  Returns (rows, outputs)."""
    import ctypes
    from field_oracle import rfc7748 as oracle_rfc7748
    path = os.path.join(ROOT, "oracle", "_ref", "libref_%s.so" % name)
    if os.path.exists(path):
        return np.arange(k.shape[0]), util.ref_rfc7748_batch(ctypes.CDLL(path), k, u)
    P = OraclePrime("M383", M383_P, a24=516287, cof=3, generator=12)
    ts = name != "M383_validate"
    return rows, np.array([np.frombuffer(oracle_rfc7748(P, k[i].tobytes(), u[i].tobytes(), twist_secure=ts),
                                         dtype=np.uint8) for i in rows]).reshape(len(rows), 48)


def _m383_batch(n):
    k, u = util.random_bytes(38301, n, 48), util.random_bytes(38302, n, 48)
    rows = [0, 1, 12, M383_P - 1, M383_P, M383_P + 1, (1 << 383) - 1, (1 << 384) - 1]
    for i, v in enumerate(rows):
        u[i] = np.frombuffer(v.to_bytes(48, "little"), dtype=np.uint8)
    k[len(rows)] = 0
    k[len(rows) + 1] = 255
    return k, u


def test_user_curve_ladder_vs_reference_build():
    from modarith_b200 import lib as mlib
    from modarith_b200.rfc7748 import rfc7748
    if not os.path.exists(mlib.extra_lib_path("M383")):
        pytest.fail("libmodarith_b200_M383.so is missing: __graft_entry__.build() builds it")
    n = (1 << 14) + 77                      # more than one chunk round of the persistent grid's queues, ragged
    k, u = _m383_batch(n)
    rows, want = _expected_m383("M383", k, u, util.sample_rows(n, 512, head=10))
    dk, du = torch.from_numpy(k).cuda(), torch.from_numpy(u).cuda()
    got = rfc7748("M383", dk, du)
    assert np.array_equal(got.cpu().numpy()[rows], want)
    # one key per thread, one inversion per key: same bytes
    lib = mlib.load_for("M383")
    out = torch.empty_like(dk)
    mlib.check(lib.mab_M383_rfc7748_perkey(dk.data_ptr(), du.data_ptr(), out.data_ptr(), n,
                                           torch.cuda.current_stream().cuda_stream), "perkey", lib)
    assert torch.equal(out, got)
    # host buffers: pageable (staged) and pinned (zero-copy)
    got = got.cpu().numpy()
    assert np.array_equal(rfc7748("M383", k, u), got)
    pk, pu = torch.from_numpy(k).pin_memory(), torch.from_numpy(u).pin_memory()
    assert np.array_equal(rfc7748("M383", pk, pu).numpy(), got)


def test_user_curve_point_validation_vs_reference_build():
    """The driver without TWIST_SECURE (rfc7748.c:228-251) -- what a user-defined curve that is not twist secure runs."""
    from modarith_b200.rfc7748 import rfc7748
    n = 1 << 12
    k, u = _m383_batch(n)
    rows, want = _expected_m383("M383_validate", k, u, util.sample_rows(n, 512, head=10))
    got = rfc7748("M383", torch.from_numpy(k).cuda(), torch.from_numpy(u).cuda(), validate=True).cpu().numpy()
    assert np.array_equal(got[rows], want)
    zero = (got == 0).all(axis=1).sum()
    assert n // 4 < zero < 3 * n // 4         # about half of all u are x-coordinates of points on the twist
