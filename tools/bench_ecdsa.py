#!/usr/bin/env python3
"""ECDSA P-256 verification rates on one GPU, in one process:

    python tools/bench_ecdsa.py [OUT.json]          # the result goes to stdout, and to OUT.json when given

At 2^18, 2^20 and 2^22 rows (160 B of input per row: from 2^20 rows up the inputs exceed the 126 MB L2), after a
warm-up of every shape, each timed with CUDA events over at least one second:
  fused      mab_NIST256_ecdsa_verify (one kernel)
  composed   the same verification chained from the existing calls (`composed` below): order-field modimp / modinv /
             modmul / modexp, the P-256 on-curve check with field calls, ecnmul2, then the compare on the device
  ecnmul2    mab_NIST256_ecnmul2 alone on the same rows
plus the limb products of one verification and the fraction of the live IMAD peak (mab_imad_peak) they reach, a CPU
baseline (OpenSSL through `cryptography`, all host cores, labelled as such), and the card name and power limit read
in the same run.  Every arm's results are checked against the expected flags of the rows.
"""
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

N_ORDER = 115792089210356248762697446949407573529996955224135760342422259061068512044369
P_FIELD = 2 ** 256 - 2 ** 224 + 2 ** 192 + 2 ** 96 - 1
B_CURVE = 0x5AC635D8AA3A93E7B3EBBD55769886BC651D06B0CC53B0F63BCE3C3E27D2604B
GX = 0x6B17D1F2E12C4247F8BCE6E563A440F277037D812DEB33A0F4A13945D898C296
GY = 0x4FE342E2FE1A7F9B8EE7EB4A7C0F9E162BCE33576B315ECECBB6406837BF51F5


def _rows(v, n, dev):
    import numpy as np
    import torch
    return torch.from_numpy(np.tile(np.frombuffer(v.to_bytes(32, "big"), dtype=np.uint8), (n, 1))).to(dev)


def composed(h, r, s, qx, qy):
    """The verification a user could chain from the library's existing calls (CUDA tensors in, CUDA bool out):
    w = s^-1, u1 = h w, u2 = r w on the order field; Q's range and curve equation on the P-256 field;
    (x, y) = ecnmul2(u1, G, u2, Q); valid iff r, s in [1, n), Q valid, R != O and x mod n == r."""
    import torch
    from modarith_b200 import Field
    from modarith_b200.ecn import ecnmul2
    n = h.shape[0]
    dev = h.device
    Fn, Fp = Field("NIST256ORDER", dev), Field("NIST256", dev)
    rm, rlt = Fn.modimp(r)
    sm, slt = Fn.modimp(s)
    hm, _ = Fn.modimp(h)
    w, u = Fn.alloc(n), Fn.alloc(n)
    Fn.modinv(sm, None, w)
    Fn.modmul(hm, w, u)
    u1 = Fn.modexp(u)
    Fn.modmul(rm, w, u)
    u2 = Fn.modexp(u)
    ok = (rlt & slt & (1 - Fn.modis0(rm)) & (1 - Fn.modis0(sm))).bool()
    x, xlt = Fp.modimp(qx)
    y, ylt = Fp.modimp(qy)
    t, t3, b = Fp.alloc(n), Fp.alloc(n), Fp.modimp(_rows(B_CURVE, n, dev))[0]
    Fp.modsqr(x, t)
    Fp.modmul(t, x, t)
    Fp.modmli(x, 3, t3)
    Fp.modsub(t, t3, t)
    Fp.modadd(t, b, t)
    Fp.modsqr(y, t3)
    ok &= (xlt & ylt & Fp.modcmp(t, t3)).bool()
    gx, gy = _rows(GX, n, dev), _rows(GY, n, dev)
    xo, yo = ecnmul2("NIST256", u1, gx, gy, u2, qx, qy)
    one = torch.zeros_like(yo)
    one[:, 31] = 1
    inf = (xo == 0).all(dim=1) & (yo == one).all(dim=1)            # ecnXXXget reports O as (0, 1), not on the curve
    xr, _ = Fn.modimp(xo)                                           # x mod n
    return ok & ~inf & (Fn.modexp(xr) == r).all(dim=1)


def products_per_verification():
    """32x32->64 limb products of one Ecdsa::verify (ecdsa_sm100.cuh), from the operation counts of the code:
    M = 64 (8x8 words), S = 36; Montgomery import / export and comparisons are one product each."""
    from modarith_b200 import lib as mlib
    M, S = 64, 36
    order = 3 * M + 2 * M + mlib.products("NIST256ORDER", "modinv") + 2 * M + 2 * M   # imports, is0, s^-1, u1 u2, export
    setpt = 2 * M + 2 * S + M + 2 * M                                 # import x y, x^3 (S + M), y^2 (S), compare
    dbl, add = 10 * M + 3 * S, 14 * M                                 # complete formulas (weierstrass_sm100.cuh)
    table = 2 * dbl + 11 * add                                        # 2P, 3P, 2Q, 3Q, nine sums a P + b Q
    dbl2 = (2 * M + S) + 2 * (4 * M + 4 * S) + 2 * M                  # dbln<2>: into Jacobian, two halved doublings, back
    loop = 128 * (dbl2 + add)
    final = 2 * (M + M + 2 * M)                                       # two candidates: import, r Z, compare (two exports)
    return order + 2 * setpt + table + loop + final


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    parts = [p.strip() for p in q.stdout.strip().splitlines()[0].split(",")] if q.returncode == 0 and q.stdout.strip() else []
    return {"name": parts[0] if parts else None, "power_limit": parts[1] if len(parts) > 1 else None,
            "max_sm_clock": parts[2] if len(parts) > 2 else None}


def signatures(count, seed=5):
    """count (message digest, r, s, qx, qy) rows signed by OpenSSL with eight keys."""
    import hashlib
    import random
    from cryptography.hazmat.primitives import hashes
    from cryptography.hazmat.primitives.asymmetric import ec, utils
    rng = random.Random(seed)
    keys = [ec.derive_private_key(rng.randrange(1, N_ORDER), ec.SECP256R1()) for _ in range(8)]
    out = []
    for i in range(count):
        k = keys[i % len(keys)]
        msg = rng.randbytes(32)
        r, s = utils.decode_dss_signature(k.sign(msg, ec.ECDSA(hashes.SHA256())))
        pn = k.public_key().public_numbers()
        out.append((int.from_bytes(hashlib.sha256(msg).digest(), "big"), r, s, pn.x, pn.y))
    return out


def cpu_baseline(seconds=2.0):
    """OpenSSL (through cryptography) verifications per second on all host cores, one process per core."""
    import multiprocessing as mp
    nproc = os.cpu_count() or 1
    with mp.get_context("spawn").Pool(nproc) as pool:
        counts = pool.map(_cpu_worker, [seconds] * nproc)
    return {"verifications_per_s": sum(counts) / seconds, "processes": nproc,
            "what": "OpenSSL ECDSA P-256 verify through python cryptography, one process per host core"}


def _cpu_worker(seconds):
    from cryptography.hazmat.primitives import hashes
    from cryptography.hazmat.primitives.asymmetric import ec
    k = ec.generate_private_key(ec.SECP256R1())
    msg = b"x" * 32
    sig = k.sign(msg, ec.ECDSA(hashes.SHA256()))
    pk = k.public_key()
    algo = ec.ECDSA(hashes.SHA256())
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        for _ in range(100):
            pk.verify(sig, msg, algo)
        n += 100
    return n


def timed(fn, min_seconds=1.0):
    import torch
    fn()
    torch.cuda.synchronize()
    reps, t = 1, 0.0
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3
        if t >= min_seconds:
            return t / reps, reps
        reps = max(reps * 2, int(reps * 1.2 * min_seconds / max(t, 1e-6)))


def main():
    import numpy as np
    import torch
    from modarith_b200 import lib as mlib
    from modarith_b200.ecdsa import verify_digest
    from modarith_b200.ecn import ecnmul2
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"card": card()}
    lib = mlib.load()
    ms, ins = ctypes.c_float(), ctypes.c_double()
    peak = 0.0
    for _ in range(3):
        mlib.check(lib.mab_imad_peak(0, 4000, 148 * 8, 256, ctypes.byref(ms), ctypes.byref(ins), None))
        peak = max(peak, ins.value / (ms.value * 1e-3))
    prods = products_per_verification()
    res["products_per_verification"] = prods
    res["imad_peak_products_per_s"] = peak
    base = signatures(1 << 14)
    cols = [np.frombuffer(b"".join(v.to_bytes(32, "big") for v in col), dtype=np.uint8).reshape(-1, 32)
            for col in zip(*base)]
    res["rows"] = {}
    for lg in (18, 20, 22):
        n = 1 << lg
        idx = np.arange(n) % len(base)
        h, r, s, qx, qy = (torch.from_numpy(np.ascontiguousarray(c[idx])).to(dev) for c in cols)
        bad = torch.from_numpy(np.arange(n) % 4 == 3).to(dev)       # every fourth row: digest changed, must fail
        h[:, 31] ^= bad.to(torch.uint8)
        want = ~bad
        u1, u2 = h, r                                              # ecnmul2 alone: any scalars do
        gx, gy = _rows(GX, n, dev), _rows(GY, n, dev)
        row = {}
        assert torch.equal(verify_digest(h, r, s, qx, qy), want), "fused: wrong flags"
        assert torch.equal(composed(h, r, s, qx, qy), want), "composed: wrong flags"
        for name, fn in (("fused", lambda: verify_digest(h, r, s, qx, qy)),
                         ("composed", lambda: composed(h, r, s, qx, qy)),
                         ("ecnmul2", lambda: ecnmul2("NIST256", u1, gx, gy, u2, qx, qy))):
            t, reps = timed(fn)
            row[name] = {"seconds_per_call": t, "reps": reps, "M_per_s": n / t / 1e6}
        row["fused"]["imad_fraction"] = n * prods / row["fused"]["seconds_per_call"] / peak
        res["rows"][str(n)] = row
        print(lg, json.dumps(row), flush=True)
        del h, r, s, qx, qy, bad, want, gx, gy
        torch.cuda.empty_cache()
    res["cpu_baseline"] = cpu_baseline()
    res["card_after"] = card()
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
