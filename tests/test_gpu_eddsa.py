"""Ed25519 verification on the GPU (mab_ED25519_eddsa_verify through modarith_b200.eddsa): every fixture row, a
2^20-row batch with seeded mutations whose expected flags follow by construction (2^14 rows also against the
oracle), the fused kernel against the same verification composed of existing calls, batch sizes, misaligned views,
host arrays, and two streams at once."""
import hashlib
import multiprocessing as mp
import os
import random
import subprocess
import sys

import numpy as np
import pytest

import eddsa_oracle as O

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
GOLDEN = os.path.join(ROOT, "tests", "golden", "eddsa_ed25519_sample.json")
pytestmark = pytest.mark.gpu
NBASE, NROWS, NKEYS = 4096, 1 << 20, 64
le = lambda v: (v % (1 << 256)).to_bytes(32, "little")


def _signatures(count, seed=25519):
    """(h, sig, pk) byte rows: signed by OpenSSL through `cryptography` when it can be imported, otherwise by the
    oracle's signer; NKEYS keys, key i % NKEYS for row i."""
    rng = random.Random(seed)
    seeds = [rng.randbytes(32) for _ in range(NKEYS)]
    try:
        from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey
        from cryptography.hazmat.primitives.serialization import Encoding, PublicFormat
        keys = [Ed25519PrivateKey.from_private_bytes(s) for s in seeds]
        pubs = [k.public_key().public_bytes(Encoding.Raw, PublicFormat.Raw) for k in keys]
        sign = lambda i, m: keys[i].sign(m)
    except ImportError:
        pubs = [O.public_key(s) for s in seeds]
        sign = lambda i, m: O.sign(seeds[i], m)
    out = []
    for i in range(count):
        msg = rng.randbytes(32)
        sig = sign(i % NKEYS, msg)
        out.append((hashlib.sha512(sig[:32] + pubs[i % NKEYS] + msg).digest(), sig, pubs[i % NKEYS]))
    return out


MUTATIONS = 8        # 0 as signed, 1 identity key with R = enc([S]B) (both valid); 2 digest bit, 3 S + L, 4 R bit,
                     # 5 key of the next row, 6 key y with no square root, 7 sign bit of R (all invalid)


@pytest.fixture(scope="module")
def batch():
    """(h [2^20, 64], sig [2^20, 64], pk [2^20, 32]) tiled from NBASE signatures, each row with a seeded mutation
    class; the expected flags."""
    base = _signatures(NBASE)
    h0, s0, k0 = (np.frombuffer(b"".join(col), dtype=np.uint8).reshape(NBASE, -1) for col in zip(*base))
    rng = np.random.Generator(np.random.PCG64(20))
    idx = rng.permutation(NROWS) % NBASE
    kind = rng.integers(0, MUTATIONS, NROWS)
    h, sig, pk = h0[idx].copy(), s0[idx].copy(), k0[idx].copy()
    prng = random.Random(7)
    ident = []                                                       # (R || S) with R = enc([S]B)
    for _ in range(64):
        S = prng.randrange(O.L)
        ident.append(O.encode(O.mul(S)) + le(S))
    ident = np.frombuffer(b"".join(ident), dtype=np.uint8).reshape(64, 64)
    m = kind == 1
    sig[m] = ident[idx[m] % 64]
    pk[m] = np.frombuffer(le(1), dtype=np.uint8)
    h[kind == 2, 5] ^= 0x20
    m = kind == 3
    s_plus_l = np.frombuffer(b"".join(le(int.from_bytes(s0[j, 32:].tobytes(), "little") + O.L) for j in range(NBASE)),
                             dtype=np.uint8).reshape(NBASE, 32)
    sig[m, 32:] = s_plus_l[idx[m]]
    sig[kind == 4, 3] ^= 0x01
    m = kind == 5
    pk[m] = k0[(idx[m] + 1) % NBASE]                                 # consecutive base rows have different keys
    y = next(y for y in range(2, 100) if O.recover_x(y, 0) is None)
    pk[kind == 6] = np.frombuffer(le(y), dtype=np.uint8)
    sig[kind == 7, 31] ^= 0x80
    return (h, sig, pk), kind < 2


def _dev(rows):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in rows]


def test_fixture_rows_through_verify_and_the_vector_runner():
    from modarith_b200 import eddsa, wire
    vs = wire.load_eddsa_vectors(GOLDEN)
    want = np.array([v.result == "valid" for v in vs])
    got = eddsa.verify([bytes.fromhex(v.msg) for v in vs], [bytes.fromhex(v.sig) for v in vs],
                       [bytes.fromhex(v.public_key) for v in vs])
    assert [(v.tc_id, v.comment) for v, g, w in zip(vs, got, want) if g != w] == []
    verified, passed = wire.run_eddsa_vectors(vs)
    assert passed.all() and np.array_equal(verified, want)
    out = subprocess.run([sys.executable, "-m", "modarith_b200.eddsa", GOLDEN], cwd=ROOT, stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True)
    assert out.returncode == 0, out.stdout[-2000:]
    assert "valid %d/%d verified, invalid %d/%d rejected" % (want.sum(), want.sum(), (~want).sum(), (~want).sum()) in out.stdout


def test_large_batch_with_mutations(batch):
    import torch
    from modarith_b200.eddsa import verify_digest
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
    assert sample.size == 1 << 14
    args = [(rows[0][i].tobytes(), rows[1][i].tobytes(), rows[2][i].tobytes()) for i in sample]
    with mp.get_context("spawn").Pool(min(16, os.cpu_count() or 1)) as pool:
        ref = pool.starmap(O.verify_digest, args, chunksize=256)
    mism = [int(i) for i, r in zip(sample, ref) if r != ok[i]]
    assert mism == [], mism[:20]


def test_fused_equals_composed_path(batch):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from bench_eddsa import composed
    from modarith_b200.eddsa import verify_digest
    rows, want = batch
    n = 1 << 16
    d = _dev([a[:n] for a in rows])
    a, b = verify_digest(*d), composed(*d)
    torch.cuda.synchronize()
    assert torch.equal(a, b) and np.array_equal(a.cpu().numpy(), want[:n])


@pytest.mark.parametrize("n", [0, 1, 127, 129, (1 << 16) + 1])
def test_batch_sizes(batch, n):
    from modarith_b200.eddsa import verify_digest
    rows, want = batch
    ok = verify_digest(*_dev([a[NROWS - n:] for a in rows])).cpu().numpy()
    assert ok.shape == (n,) and np.array_equal(ok, want[NROWS - n:])


@pytest.mark.parametrize("offset", [1, 4, 8])
def test_misaligned_views(batch, offset):
    import torch
    from modarith_b200.eddsa import verify_digest
    rows, want = batch
    n = 3000
    views = []
    for a in rows:
        w = a.shape[1]
        buf = torch.zeros(n * w + offset, dtype=torch.uint8, device="cuda")
        v = buf[offset:].view(n, w)
        v.copy_(torch.from_numpy(np.ascontiguousarray(a[:n])))
        assert v.data_ptr() % 16 == offset % 16
        views.append(v)
    assert np.array_equal(verify_digest(*views).cpu().numpy(), want[:n])


def test_host_arrays_and_cuda_tensors_agree(batch):
    import torch
    from modarith_b200.eddsa import verify_digest
    rows, want = batch
    n = 5000
    host = verify_digest(*(a[:n] for a in rows))
    assert isinstance(host, np.ndarray) and host.dtype == bool
    dev = verify_digest(*_dev([a[:n] for a in rows]))
    assert isinstance(dev, torch.Tensor) and dev.is_cuda
    assert np.array_equal(host, dev.cpu().numpy()) and np.array_equal(host, want[:n])
    out = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    r = verify_digest(*_dev([a[:n] for a in rows]), ok=out)
    assert r.data_ptr() == out.data_ptr() and np.array_equal(r.cpu().numpy(), want[:n])
    with pytest.raises(ValueError):
        verify_digest(*(a[:n] for a in rows), ok=out)
    with pytest.raises(ValueError):
        verify_digest(*_dev([a[:n] for a in rows]), ok=out[:-1])
    with pytest.raises(ValueError):
        d = _dev([a[:n] for a in rows])
        verify_digest(d[0], d[1], rows[2][:n])                        # mixed host and device


def test_two_streams_in_flight(batch):
    import torch
    from modarith_b200.eddsa import verify_digest
    rows, want = batch
    n = 1 << 16
    a, b = _dev([x[:n] for x in rows]), _dev([x[n:2 * n] for x in rows])
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        o1 = verify_digest(*a)
    with torch.cuda.stream(s2):
        o2 = verify_digest(*b)
    torch.cuda.synchronize()
    assert np.array_equal(o1.cpu().numpy(), want[:n]) and np.array_equal(o2.cpu().numpy(), want[n:2 * n])
