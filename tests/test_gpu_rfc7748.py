"""Parity of the CUDA ladder (through the C ABI) with the oracle, the golden vectors and the
reference's own C.  Bit-exact: integer/byte work."""
import numpy as np
import pytest
import torch

from field_oracle import rfc7748 as oracle_rfc7748
from modarith_b200.primes import PRIMES
import util

pytestmark = pytest.mark.gpu
CURVES = ("X25519", "X448")


def _gpu(curve, k, u):
    from modarith_b200.rfc7748 import rfc7748
    out = rfc7748(curve, torch.from_numpy(k).cuda(), torch.from_numpy(u).cuda())
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _rows(rows, nb):
    k = np.frombuffer(b"".join(bytes.fromhex(r["k"]) for r in rows), dtype=np.uint8).reshape(-1, nb).copy()
    u = np.frombuffer(b"".join(bytes.fromhex(r["u"]) for r in rows), dtype=np.uint8).reshape(-1, nb).copy()
    return k, u, [r["out"] for r in rows]


@pytest.mark.parametrize("curve", CURVES)
def test_golden_vectors(golden_rfc, curve):
    """RFC 7748 KATs, edge rows (u in {0,1,p-1,p,p+1,2^n-1,...}, k in {0,all-ones,...}) and the
    reference-generated random rows."""
    g = golden_rfc[curve]
    nb = g["nbytes"]
    v = g["rfc"]
    gen = PRIMES[curve].generator.to_bytes(nb, "little").hex()
    rows = g["edge"] + g["random"] + [
        {"k": v["sk1"], "u": gen, "out": v["pk1"]}, {"k": v["sk2"], "u": gen, "out": v["pk2"]},
        {"k": v["sk1"], "u": v["pk2"], "out": v["shared"]}, {"k": v["sk2"], "u": v["pk1"], "out": v["shared"]},
        {"k": g["demo"]["alice"], "u": gen, "out": None}]
    k, u, want = _rows(rows, nb)
    out = _gpu(curve, k, u)
    for i, w in enumerate(want):
        if w is not None:
            assert out[i].tobytes().hex() == w, (curve, i, rows[i])


@pytest.mark.parametrize("curve", CURVES)
def test_validation_tail(golden_rfc, ref_libs, curve):
    """mab_<curve>_rfc7748_validate: the driver as built without TWIST_SECURE (rfc7748.c:228-251)."""
    from modarith_b200.rfc7748 import rfc7748
    nb = PRIMES[curve].nbytes
    k, u, want = _rows(golden_rfc[curve]["validate"], nb)
    out = rfc7748(curve, torch.from_numpy(k).cuda(), torch.from_numpy(u).cuda(), validate=True).cpu().numpy()
    assert [out[i].tobytes().hex() for i in range(len(want))] == want
    key = curve + "_validate"
    if key in ref_libs:
        n = 4096
        k, u = util.random_bytes(101, n, nb), util.random_bytes(102, n, nb)
        out = rfc7748(curve, torch.from_numpy(k).cuda(), torch.from_numpy(u).cuda(), validate=True).cpu().numpy()
        assert np.array_equal(out, util.ref_rfc7748_batch(ref_libs[key], k, u))


@pytest.mark.parametrize("curve", CURVES)
def test_shared_inversion_rounds_vs_one_inversion_per_key(curve):
    """The default kernel (persistent rounds, up to four keys per thread share one inversion) against the
    plain one-key-per-thread kernel, on batch sizes that exercise K = 4, 2 and 1 rounds with ragged tails,
    with low-order inputs (zero results) scattered through the batch."""
    from modarith_b200 import lib as mlib
    l = mlib.load()
    nb = PRIMES[curve].nbytes
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    per_round = sms * (4 if curve == "X25519" else 2) * 128
    for n in (1, 31, per_round - 1, 2 * per_round + 5, 4 * per_round + 1000, 7 * per_round + 33):
        g = torch.Generator(device="cuda").manual_seed(n)
        k = torch.randint(0, 256, (n, nb), dtype=torch.uint8, device="cuda", generator=g)
        u = torch.randint(0, 256, (n, nb), dtype=torch.uint8, device="cuda", generator=g)
        u[::97] = 0                          # u = 0 -> z2 = 0 -> all-zero output
        if n > 5:
            u[5] = 0
            u[5, 0] = 1                      # u = 1: another low-order point
        a, b = torch.empty_like(k), torch.empty_like(k)
        st = torch.cuda.current_stream().cuda_stream
        mlib.check(getattr(l, "mab_%s_rfc7748" % curve)(k.data_ptr(), u.data_ptr(), a.data_ptr(), n, st))
        mlib.check(getattr(l, "mab_%s_rfc7748_perkey" % curve)(k.data_ptr(), u.data_ptr(), b.data_ptr(), n, st))
        torch.cuda.synchronize()
        assert torch.equal(a, b), (curve, n)
        assert int((a[::97] != 0).sum()) == 0


def test_demo_loop_x25519(golden_rfc):
    """rfc7748.c:main: 5000 x 2 chained calls, each output feeding the next."""
    from modarith_b200.rfc7748 import rfc7748
    d = golden_rfc["X25519"]["demo"]
    bk = torch.from_numpy(np.frombuffer(bytes.fromhex(d["key"]), dtype=np.uint8).reshape(1, 32).copy()).cuda()
    bu = torch.zeros((1, 32), dtype=torch.uint8, device="cuda")
    bu[0, 0] = 9
    bv = torch.empty_like(bu)
    for _ in range(5000):
        rfc7748("X25519", bk, bu, bv)
        rfc7748("X25519", bk, bv, bu)
    assert bu.cpu().numpy().tobytes().hex() == d["loop5000"]


@pytest.mark.parametrize("curve", CURVES)
def test_random_vs_oracle(curve):
    nb = PRIMES[curve].nbytes
    n = 300           # not a multiple of the block size: exercises the ragged tail
    k, u = util.random_bytes(7748, n, nb), util.random_bytes(7749, n, nb)
    out = _gpu(curve, k, u)
    for i in range(0, n, 3):
        assert out[i].tobytes() == oracle_rfc7748(curve, k[i].tobytes(), u[i].tobytes()), (curve, i)


@pytest.mark.parametrize("curve,n", [("X25519", 2048), ("X448", 512)])
def test_random_vs_c_oracle(curve, n):
    """A mid-size batch against the plain-C restatement (oracle/oracle.c), every element."""
    import c_oracle
    nb = PRIMES[curve].nbytes
    k, u = util.random_bytes(81, n, nb), util.random_bytes(82, n, nb)
    assert np.array_equal(_gpu(curve, k, u), c_oracle.rfc7748_batch(curve, k, u))


@pytest.mark.parametrize("curve,n", [("X25519", 1 << 16), ("X448", 1 << 14)])
def test_random_vs_reference_build(ref_libs, curve, n):
    """Every element of a large batch against the reference's own generated C (oracle/_ref); where that build is
    absent, a fixed sample of 4096 elements against the plain-C restatement (oracle/oracle.c), which
    tests/test_oracle_pinned.py pins to vectors the reference generated."""
    import c_oracle
    nb = PRIMES[curve].nbytes
    k, u = util.random_bytes(1, n, nb), util.random_bytes(2, n, nb)
    out = _gpu(curve, k, u)
    if curve in ref_libs:
        assert np.array_equal(out, util.ref_rfc7748_batch(ref_libs[curve], k, u))
    else:
        rows = util.sample_rows(n, 4096)
        assert np.array_equal(out[rows], c_oracle.rfc7748_batch(curve, k[rows], u[rows]))


@pytest.mark.parametrize("curve", CURVES)
def test_full_size_every_key_vs_reference_build(ref_libs, curve):
    """BASELINE configs 2 and 3 at their stated size: 2^20 raw PCG64(7748) key/point pairs, EVERY output
    compared byte-for-byte with rfc7748() of the reference's own generated C (rfc7748.c:156-256 with
    pseudo.py 64 X25519 / monty.py 64 X448 pasted in; OpenMP over the host cores).  Fixed rows of SURVEY.md
    8d-2 are planted at the front: u in {0, 1, p-1, p, p+1, 2^Nbits-1, generator}, k in {0, all-ones}.  Where the
    reference build is absent: the planted rows and a fixed sample of 4096 others against oracle/oracle.c."""
    import c_oracle
    P = PRIMES[curve]
    nb = P.nbytes
    n = 1 << 20
    k, u = util.random_bytes(7748, n, nb), util.random_bytes(7749, n, nb)
    row = 0
    for uv in (0, 1, P.p - 1, P.p, P.p + 1, (1 << P.nbits) - 1, P.generator):
        for kv in (0, (1 << (8 * nb)) - 1):
            u[row] = np.frombuffer((uv % (1 << (8 * nb))).to_bytes(nb, "little"), dtype=np.uint8)
            k[row] = np.frombuffer(kv.to_bytes(nb, "little"), dtype=np.uint8)
            row += 1
    out = _gpu(curve, k, u)
    if curve in ref_libs:
        want = util.ref_rfc7748_batch(ref_libs[curve], k, u)
    else:
        rows = util.sample_rows(n, 4096, head=row)
        k, u, out = k[rows], u[rows], out[rows]
        want = c_oracle.rfc7748_batch(curve, k, u)
    bad = np.nonzero((out != want).any(axis=1))[0]
    assert bad.size == 0, (curve, "first mismatching keys", bad[:8].tolist())


@pytest.mark.parametrize("curve", CURVES)
def test_empty_and_tiny_batches(curve):
    nb = PRIMES[curve].nbytes
    e = np.zeros((0, nb), dtype=np.uint8)
    assert _gpu(curve, e, e).shape == (0, nb)
    k, u = util.random_bytes(3, 1, nb), util.random_bytes(4, 1, nb)
    assert _gpu(curve, k, u)[0].tobytes() == oracle_rfc7748(curve, k[0].tobytes(), u[0].tobytes())


@pytest.mark.parametrize("curve", CURVES)
def test_misaligned_pointers(curve):
    """Byte strings that start at odd addresses take the narrow load path."""
    from modarith_b200.rfc7748 import rfc7748
    nb = PRIMES[curve].nbytes
    n = 130
    k, u = util.random_bytes(5, n, nb), util.random_bytes(6, n, nb)
    want = _gpu(curve, k, u)
    for off in (1, 4, 8):
        bufk = torch.zeros(n * nb + 16, dtype=torch.uint8, device="cuda")
        bufu = torch.zeros(n * nb + 16, dtype=torch.uint8, device="cuda")
        bufv = torch.zeros(n * nb + 16, dtype=torch.uint8, device="cuda")
        tk = bufk[off:off + n * nb].view(n, nb)
        tu = bufu[off:off + n * nb].view(n, nb)
        tv = bufv[off:off + n * nb].view(n, nb)
        tk.copy_(torch.from_numpy(k))
        tu.copy_(torch.from_numpy(u))
        rfc7748(curve, tk, tu, tv)
        assert np.array_equal(tv.cpu().numpy(), want), off


def test_full_size_properties_x25519():
    """BASELINE config 2 (2^20 keys): size-independent properties on the whole batch --
    Diffie-Hellman commutativity k1*(k2*G) == k2*(k1*G), in-place output, and agreement of the
    host-pointer pipeline with the device-pointer call; plus an oracle-checked sub-sample."""
    from modarith_b200.rfc7748 import rfc7748
    n = 1 << 20
    k1, k2 = util.random_bytes(7748, n, 32), util.random_bytes(7750, n, 32)
    g = np.zeros((n, 32), dtype=np.uint8)
    g[:, 0] = 9
    dk1, dk2, dg = (torch.from_numpy(x).cuda() for x in (k1, k2, g))
    pk1 = rfc7748("X25519", dk1, dg)
    pk2 = rfc7748("X25519", dk2, dg)
    s12 = rfc7748("X25519", dk1, pk2)
    s21 = rfc7748("X25519", dk2, pk1, pk1)                  # output aliases the u input
    torch.cuda.synchronize()
    assert torch.equal(s12, s21)
    assert int((s12 != 0).any(dim=1).sum()) == n                 # no low-order accidents
    hk1 = torch.from_numpy(k1).pin_memory()
    hg = torch.from_numpy(g).pin_memory()
    hp = rfc7748("X25519", hk1, hg)
    assert np.array_equal(np.asarray(hp), rfc7748("X25519", dk1, dg).cpu().numpy())
    p1 = pk1.cpu().numpy()      # now holds s21
    for i in range(0, n, n // 64):
        a = oracle_rfc7748("X25519", k1[i].tobytes(), g[i].tobytes())
        assert oracle_rfc7748("X25519", k2[i].tobytes(), a) == p1[i].tobytes()


def test_host_path_numpy_pageable():
    from modarith_b200.rfc7748 import x448
    n = 777
    k, u = util.random_bytes(8, n, 56), util.random_bytes(9, n, 56)
    out = x448(k, u)
    assert np.array_equal(out, _gpu("X448", k, u))


@pytest.mark.parametrize("curve,nb", [("X25519", 32), ("X448", 56)])
def test_host_path_pinned_zero_copy_and_staged_agree(curve, nb, monkeypatch):
    """Pinned buffers: the kernel reads and writes host memory itself; MAB_HOST_ZEROCOPY=0 forces the
    staged three-stream pipeline on the same buffers.  Both must equal the device-pointer call.  Ragged
    size, and a second call on a view that starts in the middle of the pinned allocation."""
    from modarith_b200.rfc7748 import rfc7748
    n = 70000 + 13
    k, u = util.random_bytes(21, n, nb), util.random_bytes(22, n, nb)
    want = _gpu(curve, k, u)
    hk, hu = torch.from_numpy(k).pin_memory(), torch.from_numpy(u).pin_memory()
    hv = torch.zeros((n, nb), dtype=torch.uint8).pin_memory()
    rfc7748(curve, hk, hu, hv)
    assert np.array_equal(hv.numpy(), want)
    hv.zero_()
    rfc7748(curve, hk[1001:], hu[1001:], hv[1001:])
    assert np.array_equal(hv.numpy()[1001:], want[1001:]) and not hv.numpy()[:1001].any()
    monkeypatch.setenv("MAB_HOST_ZEROCOPY", "0")
    hv.zero_()
    rfc7748(curve, hk, hu, hv)
    assert np.array_equal(hv.numpy(), want)


def test_cross_check_openssl():
    """Independent implementation (OpenSSL through `cryptography`), canonical inputs only."""
    x = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.x25519")
    n = 64
    k, u = util.random_bytes(10, n, 32), util.random_bytes(11, n, 32)
    out = _gpu("X25519", k, u)
    for i in range(n):
        priv = x.X25519PrivateKey.from_private_bytes(k[i].tobytes())
        try:
            want = priv.exchange(x.X25519PublicKey.from_public_bytes(u[i].tobytes()))
        except Exception:
            continue            # OpenSSL rejects all-zero shared secrets
        assert out[i].tobytes() == want


def test_many_outstanding_launches_on_several_streams():
    """More launches in flight than the library has work-counter slots (256), spread over several streams: a slot
    is only handed out again after the launch that used it last has finished (event per slot, ADVICE r1)."""
    from modarith_b200.rfc7748 import rfc7748
    nb, n = 32, 2500
    k, u = util.random_bytes(61, n, nb), util.random_bytes(62, n, nb)
    want = _gpu("X25519", k, u)
    dk, du = torch.from_numpy(k).cuda(), torch.from_numpy(u).cuda()
    streams = [torch.cuda.Stream() for _ in range(4)]
    outs = []
    for i in range(300):
        s = streams[i % 4]
        with torch.cuda.stream(s):
            outs.append(rfc7748("X25519", dk, du))
    torch.cuda.synchronize()
    for i in (0, 1, 2, 3, 150, 255, 256, 257, 299):
        assert np.array_equal(outs[i].cpu().numpy(), want), i


def test_release_workspaces_then_reuse():
    from modarith_b200 import lib as mlib
    from modarith_b200.rfc7748 import rfc7748
    k, u = util.random_bytes(63, 777, 32), util.random_bytes(64, 777, 32)
    want = _gpu("X25519", k, u)
    assert np.array_equal(rfc7748("X25519", k, u), want)          # host route: creates the per-device workspace
    torch.cuda.synchronize()
    mlib.load().mab_release_workspaces()
    assert np.array_equal(_gpu("X25519", k, u), want)
    assert np.array_equal(rfc7748("X25519", k, u), want)
