"""Parity of the batched field API (C ABI, limb planes on the GPU) with the oracle, the golden
vectors produced by the reference's generated C, and oracle/_ref at larger sizes."""
import random

import numpy as np
import pytest
import torch

from field_oracle import FieldOracle
from modarith_b200.primes import ALL_PRIMES as PRIMES
import util

pytestmark = pytest.mark.gpu
NAMES = list(PRIMES)


def _field(name):
    from modarith_b200 import Field
    return Field(name)


def _bytes(t):
    return t.cpu().numpy()


@pytest.mark.parametrize("name", NAMES)
def test_field_golden(golden_field, name):
    g = golden_field[name]
    F = _field(name)
    nb = g["nbytes"]
    a = torch.from_numpy(np.frombuffer(bytes.fromhex("".join(g["a"])), dtype=np.uint8).reshape(-1, nb).copy()).cuda()
    b = torch.from_numpy(np.frombuffer(bytes.fromhex("".join(g["b"])), dtype=np.uint8).reshape(-1, nb).copy()).cuda()
    x, st = F.modimp(a)
    y, _ = F.modimp(b)
    assert st.cpu().tolist() == g["ops"]["id"]["status"]
    n = x.shape[1]
    r = F.alloc(n)

    def check(op):
        out = _bytes(F.modexp(r))
        got = [out[i].tobytes().hex() for i in range(n)]
        assert got == g["ops"][op]["out"], (name, op)

    F.modmul(x, y, r); check("mul")
    F.modsqr(x, r); check("sqr")
    F.modinv(x, None, r); check("inv")
    F.modsqrt(x, None, r); check("sqrt")
    F.modadd(x, y, r); check("add")
    F.modsub(x, y, r); check("sub")
    F.modneg(x, r); check("neg")
    F.modpro(x, r); check("pro")
    F.modcpy(x, r); check("id")
    F.modmli(x, g["mli_int"], r); check("mli")
    F.modcpy(x, r); F.modhaf(r); check("haf")
    assert F.modqr(None, x).cpu().tolist() == g["ops"]["qr"]["status"]


@pytest.mark.parametrize("name", NAMES)
def test_every_api_function_vs_oracle(name):
    F = _field(name)
    O = FieldOracle(name)
    p = O.p
    rng = random.Random(2)
    xs = [0, 1, 2, p - 1, p - 2, (p + 1) // 2, 4, 9] + [rng.randrange(p) for _ in range(200)]
    ys = [rng.randrange(p) for _ in xs]
    n = len(xs)
    x, y = F.from_ints(xs), F.from_ints(ys)
    r, h = F.alloc(n), F.alloc(n)
    assert F.to_ints(x) == xs
    F.modpro(x, h)
    assert F.to_ints(h) == [O.modpro(v) for v in xs]
    F.modinv(x, h, r)
    assert F.to_ints(r) == [O.modinv(v) for v in xs]
    F.modsqrt(x, h, r)
    assert F.to_ints(r) == [O.modsqrt(v) for v in xs]
    assert F.modqr(h, x).cpu().tolist() == [O.modqr(None, v) for v in xs]
    assert F.modis1(x).cpu().tolist() == [int(v == 1) for v in xs]
    assert F.modis0(x).cpu().tolist() == [int(v == 0) for v in xs]
    F.modcpy(x, r); F.modnsqr(r, 7)
    assert F.to_ints(r) == [pow(v, 128, p) for v in xs]
    F.modone(r); assert F.to_ints(r) == [1] * n
    F.modzer(r); assert F.to_ints(r) == [0] * n
    F.modint(12345, r); assert F.to_ints(r) == [12345] * n
    # nres / redc: plain side is the canonical value as little-endian 32-bit word planes
    plain = F.alloc(n)
    F.redc(x, plain)
    pw = plain.cpu().numpy().astype(np.uint32)
    assert [sum(int(pw[j, i]) << (32 * j) for j in range(F.Nlimbs)) for i in range(n)] == xs
    F.nres(plain, r)
    assert F.to_ints(r) == xs
    bits = torch.tensor([i & 1 for i in range(n)], dtype=torch.int32, device="cuda")
    g_, f_ = x.clone(), y.clone()
    F.modcsw(bits, g_, f_)
    assert F.to_ints(g_) == [ys[i] if i & 1 else xs[i] for i in range(n)]
    assert F.to_ints(f_) == [xs[i] if i & 1 else ys[i] for i in range(n)]
    f_ = y.clone()
    F.modcmv(bits, x, f_)
    assert F.to_ints(f_) == [xs[i] if i & 1 else ys[i] for i in range(n)]
    F.modcpy(x, r); F.modshl(5, r)
    assert F.to_ints(r) == [O.modshl(5, v) for v in xs]
    F.modcpy(x, r); F.modhaf(r)
    assert F.to_ints(r) == [O.modhaf(v) for v in xs]
    assert F.modsign(x).cpu().tolist() == [v & 1 for v in xs]
    assert F.modcmp(x, y).cpu().tolist() == [int(a == b) for a, b in zip(xs, ys)]
    assert F.modcmp(x, x).cpu().tolist() == [1] * n
    F.modcpy(x, r)
    assert F.modfsb(r).cpu().tolist() == [1] * n
    for rr in (0, 31, 32, 200, O.P.nbits - 1, 8 * O.nbytes - 1, 8 * O.nbytes):
        F.mod2r(rr, r)
        assert F.to_ints(r)[:3] == [O.mod2r(rr)] * 3
    if name in ("X25519", "X448"):   # modshr acts on the stored value (plain for these moduli)
        F.modcpy(x, r)
        out = F.modshr(8, r).cpu().tolist()
        assert list(zip(F.to_ints(r), out)) == [O.modshr(8, v) for v in xs]


@pytest.mark.parametrize("name", NAMES)
def test_shared_chain_modinv(name):
    """modinv shares one progenitor chain among 8 elements per thread: same values as one chain per
    element, zeros (and p, 2p-ish inputs that reduce to zero) anywhere in the batch, ragged sizes, in place."""
    F = _field(name)
    p = PRIMES[name].p
    rng = random.Random(8)
    for n in (1, 7, 129, 1024 + 3, 5000):
        xs = [rng.randrange(p) for _ in range(n)]
        for i in range(0, n, 11):
            xs[i] = 0
        if n > 3:
            xs[3] = p                      # imports as zero
        x = F.from_ints(xs)
        want = [pow(v % p, -1, p) if v % p else 0 for v in xs]
        z = F.alloc(n)
        F.modinv(x, None, z)
        assert F.to_ints(z) == want
        F.modinv_perelement(x, z)
        assert F.to_ints(z) == want
        F.modinv(x, None, x)               # in place
        assert F.to_ints(x) == want


@pytest.mark.parametrize("name", NAMES)
def test_aliasing_and_pitch(name):
    """Outputs may alias inputs (pseudo.py:1832-1845); planes may be a window of a wider pitch."""
    F = _field(name)
    O = FieldOracle(name)
    p = O.p
    rng = random.Random(3)
    n = 100
    xs, ys = [rng.randrange(p) for _ in range(n)], [rng.randrange(p) for _ in range(n)]
    x, y = F.from_ints(xs), F.from_ints(ys)
    F.modmul(x, y, x)
    assert F.to_ints(x) == [a * b % p for a, b in zip(xs, ys)]
    F.modadd(y, y, y)
    assert F.to_ints(y) == [2 * b % p for b in ys]
    F.modinv(y, None, y)
    assert F.to_ints(y) == [pow(2 * b, -1, p) for b in ys]
    wide = torch.zeros((F.Nlimbs, 4 * n), dtype=torch.int32, device="cuda")
    a, b, c = wide[:, 0:n], wide[:, n:2 * n], wide[:, 3 * n:4 * n]
    a.copy_(F.from_ints(xs)); b.copy_(F.from_ints(ys))
    F.modmul(a, b, c)
    assert F.to_ints(c.contiguous()) == [u * v % p for u, v in zip(xs, ys)]
    assert int(wide[:, 2 * n:3 * n].abs().sum()) == 0


@pytest.mark.parametrize("name", NAMES)
def test_reference_selftest_sequence(name):
    """The generator's own ctypes self-test (pseudo.py:1762-1855), 1000 random x,y, run through the
    batched ABI: redc(...) must equal ((x-y)(x+y))^-2.  (modshl/modshr pair omitted: DESIGN.md.)"""
    F = _field(name)
    p = PRIMES[name].p
    rng = random.Random(4)
    lim = min(2 * p, 1 << (8 * F.Nbytes))
    xs, ys = [rng.randrange(lim) for _ in range(1000)], [rng.randrange(lim) for _ in range(1000)]
    x, y = F.from_ints(xs), F.from_ints(ys)
    t, z = F.alloc(1000), F.alloc(1000)
    F.modadd(x, y, t)
    F.modsub(x, y, z)
    F.modmul(t, z, x)
    F.modsqr(x, z)
    F.modinv(z, None, z)
    F.modsqrt(z, None, z)
    F.modsqr(z, z)
    F.modhaf(z)
    F.modadd(z, z, z)
    got = F.to_ints(z)
    for i in range(1000):
        w = (xs[i] - ys[i]) * (xs[i] + ys[i]) % p
        assert got[i] == (pow(w * w % p, -1, p) if w else 0)


@pytest.mark.parametrize("name", NAMES)
def test_large_batch_vs_reference_build(ref_libs, name):
    """Six field operations on 2^15 elements against the reference's own generated C (oracle/_ref); where that build
    is absent, the corner rows and a fixed sample of 2048 others against the plain-C restatement (oracle/oracle.c),
    which tests/test_oracle_pinned.py pins to vectors the reference generated."""
    import c_oracle
    key = name + "_generic" if name in ("X25519", "X448") else name
    F = _field(name)
    nb = F.Nbytes
    n = 1 << 15
    a, b = util.random_bytes(41, n, nb), util.random_bytes(42, n, nb)
    # explicit corner rows (SURVEY.md 8d config 4): p-1, p, p+1, 2^(8*Nbytes)-1, 0, 1
    p = PRIMES[name].p
    for i, v in enumerate([p - 1, p, p + 1, (1 << (8 * nb)) - 1, 0, 1]):
        a[i] = np.frombuffer(v.to_bytes(nb, "big"), dtype=np.uint8)
    x, st = F.modimp(torch.from_numpy(a).cuda())
    y, _ = F.modimp(torch.from_numpy(b).cuda())
    r = F.alloc(n)
    for op in ("mul", "sqr", "inv", "sqrt", "add", "sub"):
        if key in ref_libs:
            rows = np.arange(n)
            want, wst = util.ref_field_batch(ref_libs[key], op, a, b if op in ("mul", "add", "sub") else None)
        else:
            rows = util.sample_rows(n, 2048, head=6)
            want, wst = c_oracle.field_batch(name, op, a[rows], b[rows] if op in ("mul", "add", "sub") else None)
        if op == "mul": F.modmul(x, y, r)
        if op == "sqr": F.modsqr(x, r)
        if op == "inv": F.modinv(x, None, r)
        if op == "sqrt": F.modsqrt(x, None, r)
        if op == "add": F.modadd(x, y, r)
        if op == "sub": F.modsub(x, y, r)
        assert np.array_equal(_bytes(F.modexp(r))[rows], want), (name, op)
        assert np.array_equal(st.cpu().numpy()[rows], wst)


def test_p256_full_size_properties():
    """BASELINE config 4 (2^24 P-256 elements): size-independent identities on the whole batch:
    a * a^-1 == 1 (a != 0), sqrt(a^2)^2 == a^2, (a+b)-b == a, a*b == b*a."""
    F = _field("NIST256")
    n = 1 << 24
    gen = torch.Generator(device="cuda").manual_seed(256)
    a8 = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=gen)
    b8 = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=gen)
    x, _ = F.modimp(a8)
    y, _ = F.modimp(b8)
    del a8, b8
    r, s = F.alloc(n), F.alloc(n)
    F.modinv(x, None, r)
    F.modmul(r, x, r)
    assert int(F.modis1(r).sum()) + int(F.modis0(x).sum()) == n
    F.modsqr(x, r)
    F.modsqrt(r, None, s)
    F.modsqr(s, s)
    assert int(F.modcmp(r, s).sum()) == n
    F.modadd(x, y, r)
    F.modsub(r, y, r)
    assert int(F.modcmp(r, x).sum()) == n
    F.modmul(x, y, r)
    F.modmul(y, x, s)
    assert int(F.modcmp(r, s).sum()) == n


def test_p256_full_size_sample_vs_reference_build(ref_libs):
    """BASELINE config 4 at its stated size (2^24 P-256 elements through modimp -> op -> modexp) with a 2^20
    sub-sample -- one contiguous block of 2^19 elements plus every 32nd element of the batch -- compared
    byte-for-byte with the reference's generated C (monty.py 64 NIST256) for modmul, modsqr, modinv, modsqrt,
    modadd and modsub, modimp status included.  Corner rows of SURVEY.md 8d-4 are planted inside the sample:
    p-1, p, p+1, 2^256-1, 0, 1.  Where the reference build is absent, the corner rows and a fixed sample of 2048
    other sample rows are compared with the plain-C restatement (oracle/oracle.c) instead."""
    import c_oracle
    F = _field("NIST256")
    p = PRIMES["NIST256"].p
    n = 1 << 24
    gen = torch.Generator(device="cuda").manual_seed(2561)
    a8 = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=gen)
    b8 = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=gen)
    base = 5 * (1 << 20) + 17                             # contiguous block, not block-aligned
    idx = torch.cat([torch.arange(base, base + (1 << 19), device="cuda"), torch.arange(0, n, 32, device="cuda")])
    assert idx.numel() == 1 << 20
    for j, v in enumerate([p - 1, p, p + 1, (1 << 256) - 1, 0, 1]):
        a8[base + j] = torch.from_numpy(np.frombuffer(v.to_bytes(32, "big"), dtype=np.uint8).copy()).cuda()
    x, st = F.modimp(a8)
    y, _ = F.modimp(b8)
    if "NIST256" not in ref_libs:
        idx = idx[torch.from_numpy(util.sample_rows(idx.numel(), 2048, head=6)).cuda()]
    a, b = a8[idx].cpu().numpy(), b8[idx].cpu().numpy()
    del a8, b8
    r = F.alloc(n)
    out = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    for op in ("mul", "sqr", "inv", "sqrt", "add", "sub"):
        if op == "mul": F.modmul(x, y, r)
        if op == "sqr": F.modsqr(x, r)
        if op == "inv": F.modinv(x, None, r)
        if op == "sqrt": F.modsqrt(x, None, r)
        if op == "add": F.modadd(x, y, r)
        if op == "sub": F.modsub(x, y, r)
        F.modexp(r, out)
        want, wst = (util.ref_field_batch(ref_libs["NIST256"], op, a, b if op in ("mul", "add", "sub") else None)
                     if "NIST256" in ref_libs else c_oracle.field_batch("NIST256", op, a, b if op in ("mul", "add", "sub") else None))
        got = out[idx].cpu().numpy()
        bad = np.nonzero((got != want).any(axis=1))[0]
        assert bad.size == 0, (op, "first mismatching sample rows", bad[:8].tolist())
        assert np.array_equal(st[idx].cpu().numpy(), wst)


@pytest.mark.parametrize("name", NAMES)
def test_modfsb_on_noncanonical_stored_values(name):
    """modfsb (pseudo.py:272-283) returns 0 and reduces when the stored value is >= p.  Stored values >= p
    exist for the weakly reduced plans (2^255-19: anything below 2^256; 2^448-2^224-1: below 2^448) and are
    planted here as raw limb planes; the fully reduced Montgomery plans only ever hold values below p, so
    for them the flag is 1 and the value unchanged -- both asserted."""
    from modarith_b200.gen.plan import make_plan
    F = _field(name)
    P = PRIMES[name]
    plan = make_plan(P)
    p, L = P.p, F.Nlimbs
    rng = random.Random(5)
    top = plan.bound
    vals = [0, 1, p - 1] + [rng.randrange(p) for _ in range(40)]
    if top > p:
        vals += [p, p + 1, top - 1, (p + top) // 2] + [rng.randrange(p, top) for _ in range(40)]
    planes = np.zeros((L, len(vals)), dtype=np.uint32)
    for i, v in enumerate(vals):
        for j in range(L):
            planes[j, i] = (v >> (32 * j)) & 0xFFFFFFFF
    x = torch.from_numpy(planes.view(np.int32)).cuda()
    flags = F.modfsb(x).cpu().tolist()
    assert flags == [int(v < p) for v in vals]
    got = x.cpu().numpy().view(np.uint32).astype(object)
    back = [sum(int(got[j, i]) << (32 * j) for j in range(L)) for i in range(len(vals))]
    assert back == [v % p for v in vals]
    if top > p:
        assert 0 in flags


@pytest.mark.parametrize("name", ["NIST256", "SECP256K1", "NIST256ORDER"])
def test_modshr_montgomery_moduli(name):
    """modshr on the Montgomery moduli, used the way the reference uses it (modexp / modhaf / rfc7748.c:250:
    on a canonical plain value): redc first, shift the plain words, compare value and shifted-out bits."""
    F = _field(name)
    O = FieldOracle(name)
    p = O.p
    rng = random.Random(6)
    xs = [0, 1, p - 1, p - 2, 255, 256] + [rng.randrange(p) for _ in range(300)]
    x = F.from_ints(xs)
    plain = F.alloc(len(xs))
    for sh in (1, 8, 31):
        F.redc(x, plain)
        out = F.modshr(sh, plain).cpu().tolist()
        pw = plain.cpu().numpy().view(np.uint32).astype(object)
        got = [sum(int(pw[j, i]) << (32 * j) for j in range(F.Nlimbs)) for i in range(len(xs))]
        assert got == [v >> sh for v in xs]
        assert out == [v & ((1 << sh) - 1) for v in xs]
        assert [(g, o) for g, o in zip(got, out)] == [O.modshr(sh, v) for v in xs]


def test_unsaturated_comparison_kernel():
    """csrc/mab_unsat29.cuh (the reference's radix-2^29 x 9 plan, kept only to be measured against the
    saturated plan) computes a * b^k mod 2^255-19."""
    from modarith_b200 import lib as mlib
    l = mlib.load()
    p = PRIMES["X25519"].p
    rng = random.Random(29)
    n, iters = 300, 37
    xs, ys = [rng.randrange(p) for _ in range(n)], [rng.randrange(p) for _ in range(n)]

    def planes(vals):
        a = np.zeros((9, n), dtype=np.uint32)
        for i, v in enumerate(vals):
            for k in range(9):
                a[k, i] = (v >> (29 * k)) & ((1 << 29) - 1)
        return torch.from_numpy(a.view(np.int32)).cuda()

    a, b = planes(xs), planes(ys)
    c = torch.empty_like(a)
    mlib.check(l.mab_probe_unsat29_modmul(a.data_ptr(), b.data_ptr(), c.data_ptr(), iters, n, n,
                                          torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    out = c.cpu().numpy().view(np.uint32).astype(object)
    for i in range(n):
        got = sum(int(out[k, i]) << (29 * k) for k in range(9)) % p
        assert got == xs[i] * pow(ys[i], iters, p) % p
