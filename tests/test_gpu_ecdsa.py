"""ECDSA P-256 verification on the GPU (mab_NIST256_ecdsa_verify through modarith_b200.ecdsa): every fixture row,
a 2^20-row batch with seeded mutations whose expected flags follow by construction (a sample of 2^14 rows also
against the oracle), the fused kernel against the same verification composed of existing calls, batch sizes,
misaligned views, host arrays, and two streams at once."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import ecdsa_oracle as O

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
GOLDEN = [os.path.join(ROOT, "tests", "golden", f) for f in ("ecdsa_secp256r1_sha256_sample.json",
                                                             "ecdsa_secp256r1_sha256_p1363_sample.json")]
pytestmark = pytest.mark.gpu
NBASE, NROWS = 1 << 14, 1 << 20
be = lambda v: (v % (1 << 256)).to_bytes(32, "big")


def _signatures(count, seed=14):
    """(h, r, s, qx, qy) integers: signed by OpenSSL through `cryptography` when it can be imported, otherwise by the
    oracle's signer; 32 keys, key i % 32 for row i."""
    rng = random.Random(seed)
    ds = [rng.randrange(1, O.N) for _ in range(32)]
    try:
        import hashlib
        from cryptography.hazmat.primitives import hashes
        from cryptography.hazmat.primitives.asymmetric import ec, utils
    except ImportError:
        keys = [O.public_key(d) for d in ds]
        out = []
        for i in range(count):
            h = rng.randrange(1 << 256)
            r, s = O.sign(ds[i % 32], h, rng.randrange(1, O.N))
            out.append((h, r, s) + keys[i % 32])
        return out
    sk = [ec.derive_private_key(d, ec.SECP256R1()) for d in ds]
    pub = [k.public_key().public_numbers() for k in sk]
    out = []
    for i in range(count):
        msg = rng.randbytes(32)
        r, s = utils.decode_dss_signature(sk[i % 32].sign(msg, ec.ECDSA(hashes.SHA256())))
        out.append((int.from_bytes(hashlib.sha256(msg).digest(), "big"), r, s, pub[i % 32].x, pub[i % 32].y))
    return out


MUTATIONS = 8        # 0 as signed, 1 s -> n - s (both valid); 2 digest bit, 3 r = 0, 4 s = n, 5 key of the next row,
                     # 6 qy bit (off the curve), 7 r bit (all invalid)


@pytest.fixture(scope="module")
def batch():
    """[5, 2^20, 32] rows tiled from 2^14 signatures, each with a seeded mutation class; the expected flags."""
    base = _signatures(NBASE)
    cols = np.stack([np.frombuffer(b"".join(be(v) for v in col), dtype=np.uint8).reshape(-1, 32) for col in zip(*base)])
    neg_s = np.frombuffer(b"".join(be(O.N - row[2]) for row in base), dtype=np.uint8).reshape(-1, 32)
    rng = np.random.Generator(np.random.PCG64(20))
    idx = rng.permutation(NROWS) % NBASE
    kind = rng.integers(0, MUTATIONS, NROWS)
    rows = cols[:, idx].copy()
    h, r, s, qx, qy = rows
    m = kind == 1
    s[m] = neg_s[idx[m]]
    h[kind == 2, 31] ^= 1
    r[kind == 3] = 0
    s[kind == 4] = np.frombuffer(be(O.N), dtype=np.uint8)
    m = kind == 5
    nxt = (idx[m] + 1) % NBASE                                        # consecutive base rows have different keys
    qx[m], qy[m] = cols[3, nxt], cols[4, nxt]
    qy[kind == 6, 31] ^= 1
    r[kind == 7, 31] ^= 0x10
    return rows, kind < 2


def _dev(rows):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in rows]


def _oracle_row(rows, i):
    v = [int.from_bytes(rows[k][i].tobytes(), "big") for k in range(5)]
    return O.verify(v[0], v[1], v[2], (v[3], v[4]))


def test_fixture_rows_through_verify_and_the_vector_runner():
    from modarith_b200 import ecdsa, wire
    for path in GOLDEN:
        vs = wire.load_ecdsa_vectors(path)
        want = np.array([v.result == "valid" for v in vs])
        got = np.zeros(len(vs), dtype=bool)
        for h, enc in sorted({(v.hash or "", v.encoding) for v in vs}):
            idx = [i for i, v in enumerate(vs) if (v.hash or "", v.encoding) == (h, enc)]
            got[idx] = ecdsa.verify([bytes.fromhex(vs[i].msg) for i in idx], [bytes.fromhex(vs[i].sig) for i in idx],
                                    [bytes.fromhex(vs[i].public_key) for i in idx], hash=h or None, encoding=enc)
        assert [(v.tc_id, v.comment) for v, g, w in zip(vs, got, want) if g != w] == []
        verified, passed = wire.run_ecdsa_vectors(vs)
        assert passed.all() and np.array_equal(verified, want)
        out = subprocess.run([sys.executable, "-m", "modarith_b200.ecdsa", path], cwd=ROOT, stdout=subprocess.PIPE,
                             stderr=subprocess.STDOUT, text=True)
        assert out.returncode == 0, out.stdout[-2000:]
        assert "valid %d/%d verified" % (want.sum(), want.sum()) in out.stdout


def test_large_batch_with_mutations(batch):
    import torch
    from modarith_b200.ecdsa import verify_digest
    rows, want = batch
    ok = verify_digest(*_dev(rows))
    torch.cuda.synchronize()
    ok = ok.cpu().numpy()
    assert ok.dtype == bool and ok.shape == (NROWS,)
    bad = np.nonzero(ok != want)[0]
    assert bad.size == 0, bad[:20]
    # 2^14 rows against the oracle: a contiguous block, a strided sample, the batch tail
    sample = np.concatenate([np.arange(0, 6000), np.arange(6000, NROWS - 4384, (NROWS - 10384) // 6000)[:6000],
                             np.arange(NROWS - 4384, NROWS)])
    assert sample.size == NBASE
    for i in sample:
        assert _oracle_row(rows, i) == ok[i], i


def test_fused_equals_composed_path(batch):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from bench_ecdsa import composed
    from modarith_b200.ecdsa import verify_digest
    rows, want = batch
    n = 1 << 16
    d = _dev(rows[:, :n])
    a, b = verify_digest(*d), composed(*d)
    torch.cuda.synchronize()
    assert torch.equal(a, b) and np.array_equal(a.cpu().numpy(), want[:n])


@pytest.mark.parametrize("n", [0, 1, 127, 129, (1 << 17) + 3])
def test_batch_sizes(batch, n):
    from modarith_b200.ecdsa import verify_digest
    rows, want = batch
    ok = verify_digest(*_dev(rows[:, NROWS - n:])).cpu().numpy()
    assert ok.shape == (n,) and np.array_equal(ok, want[NROWS - n:])


@pytest.mark.parametrize("offset", [1, 4])
def test_misaligned_views(batch, offset):
    import torch
    from modarith_b200.ecdsa import verify_digest
    rows, want = batch
    n = 3000
    views = []
    for a in rows[:, :n]:
        buf = torch.zeros(n * 32 + offset, dtype=torch.uint8, device="cuda")
        v = buf[offset:].view(n, 32)
        v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        assert v.data_ptr() % 16 == offset % 16
        views.append(v)
    assert np.array_equal(verify_digest(*views).cpu().numpy(), want[:n])


def test_host_arrays_and_cuda_tensors_agree(batch):
    import torch
    from modarith_b200.ecdsa import verify_digest
    rows, want = batch
    n = 5000
    host = verify_digest(*rows[:, :n])
    assert isinstance(host, np.ndarray) and host.dtype == bool
    dev = verify_digest(*_dev(rows[:, :n]))
    assert isinstance(dev, torch.Tensor) and dev.is_cuda
    assert np.array_equal(host, dev.cpu().numpy()) and np.array_equal(host, want[:n])
    out = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    r = verify_digest(*_dev(rows[:, :n]), ok=out)
    assert r.data_ptr() == out.data_ptr() and np.array_equal(r.cpu().numpy(), want[:n])
    with pytest.raises(ValueError):
        verify_digest(*rows[:, :n], ok=out)
    with pytest.raises(ValueError):
        verify_digest(*_dev(rows[:, :n]), ok=out[:-1])
    with pytest.raises(ValueError):
        verify_digest(rows[0, :n, :31], *rows[1:, :n])


def test_two_streams_in_flight(batch):
    import torch
    from modarith_b200.ecdsa import verify_digest
    rows, want = batch
    n = 1 << 16
    a, b = _dev(rows[:, :n]), _dev(rows[:, n:2 * n])
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        o1 = verify_digest(*a)
    with torch.cuda.stream(s2):
        o2 = verify_digest(*b)
    torch.cuda.synchronize()
    assert np.array_equal(o1.cpu().numpy(), want[:n]) and np.array_equal(o2.cpu().numpy(), want[n:2 * n])
