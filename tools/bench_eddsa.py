#!/usr/bin/env python3
"""Ed25519 verification rates on one GPU, in one process:

    python tools/bench_eddsa.py [OUT.json]          # the result goes to stdout, and to OUT.json when given

At 2^18, 2^20 and 2^22 rows (160 B of input per row: from 2^20 rows up the inputs exceed the 126 MB L2), after a
warm-up of every shape, each timed over at least one second:
  fused      mab_ED25519_eddsa_verify (one kernel), CUDA events
  composed   the same verification from the existing calls (`composed` below): S < L, the key decoding and
             k = h mod L on the host (there is no device call for the order field of Ed25519), ecnmul2 on the
             device, encode-and-compare on the device; host clock around the whole call, ending in a synchronise
  ecnmul2    mab_ED25519_ecnmul2 alone on the same rows, CUDA events
plus the limb products of one verification (and of ecnmul2, counted the same way) and the fraction of the live IMAD
peak (mab_imad_peak) they reach, a CPU baseline (OpenSSL through `cryptography`, one process per logical CPU,
labelled as such), and the card name and power limit read in the same run.  Every arm's results are checked
against the expected flags of the rows.
"""
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

P_FIELD = 2 ** 255 - 19
L_ORDER = 2 ** 252 + 27742317777372353535851937790883648493
D_CURVE = 0x52036CEE2B6FFE738CC740797779E89800700A4D4141D8AB75EB4DCA135978A3
GX = 0x216936D3CD6E53FEC0A4E231FDD6DC5C692CC7609525A7B2C9562D608F25D51A
GY = 0x6666666666666666666666666666666666666666666666666666666666666658
SQRT_M1 = pow(2, (P_FIELD - 1) // 4, P_FIELD)


def _decode_key(enc: bytes):
    """RFC 8032 5.1.3, strict, on the host: (x, y) or None."""
    v = int.from_bytes(enc, "little")
    y, sign = v & ((1 << 255) - 1), v >> 255
    if y >= P_FIELD:
        return None
    u, w = (y * y - 1) % P_FIELD, (D_CURVE * y * y + 1) % P_FIELD
    x2 = u * pow(w, -1, P_FIELD) % P_FIELD
    x = pow(x2, (P_FIELD + 3) // 8, P_FIELD)
    if (x * x - x2) % P_FIELD:
        x = x * SQRT_M1 % P_FIELD
    if (x * x - x2) % P_FIELD or (x == 0 and sign):
        return None
    return (P_FIELD - x if (x & 1) != sign else x), y


def host_prepare(h, sig, pk):
    """The host half of the composed path (numpy [n, 64] / [n, 64] / [n, 32] uint8 in): e = S, f = k = h mod L and
    -A as big-endian [n, 32] rows for ecnmul2, and ok[n] = S < L and A decodes.  Keys are decoded once per distinct
    key."""
    import numpy as np
    n = h.shape[0]
    keys, inv = np.unique(pk, axis=0, return_inverse=True)
    dec = [_decode_key(k.tobytes()) for k in keys]
    kx = np.zeros((len(keys), 32), dtype=np.uint8)
    ky = np.zeros((len(keys), 32), dtype=np.uint8)
    kok = np.zeros(len(keys), dtype=bool)
    for j, d in enumerate(dec):
        if d is not None:
            kx[j] = np.frombuffer(((-d[0]) % P_FIELD).to_bytes(32, "big"), dtype=np.uint8)
            ky[j] = np.frombuffer(d[1].to_bytes(32, "big"), dtype=np.uint8)
            kok[j] = True
    inv = inv.reshape(-1)
    s_le = sig[:, 32:]
    e = np.ascontiguousarray(s_le[:, ::-1])
    hb = h.tobytes()
    f = np.frombuffer(b"".join((int.from_bytes(hb[64 * i:64 * i + 64], "little") % L_ORDER).to_bytes(32, "big")
                               for i in range(n)), dtype=np.uint8).reshape(n, 32).copy()
    lt = np.array([int.from_bytes(s_le[i].tobytes(), "little") < L_ORDER for i in range(n)], dtype=bool)
    return e, f, kx[inv], ky[inv], lt & kok[inv]


def composed(h, sig, pk):
    """The verification a user could chain from the library's existing calls (CUDA tensors in, CUDA bool out): host
    preparation (host_prepare), R' = (x, y) = ecnmul2(S, B, k, -A) on the device, then encode(R') == R on the
    device."""
    import numpy as np
    import torch
    from modarith_b200.ecn import ecnmul2
    dev = h.device
    n = h.shape[0]
    e, f, x2, y2, ok = host_prepare(h.cpu().numpy(), sig.cpu().numpy(), pk.cpu().numpy())
    gx = torch.from_numpy(np.tile(np.frombuffer(GX.to_bytes(32, "big"), dtype=np.uint8), (n, 1))).to(dev)
    gy = torch.from_numpy(np.tile(np.frombuffer(GY.to_bytes(32, "big"), dtype=np.uint8), (n, 1))).to(dev)
    t = lambda a: torch.from_numpy(a).to(dev)
    xo, yo = ecnmul2("ED25519", t(e), gx, gy, t(f), t(x2), t(y2))
    enc = yo.flip(1).clone()                                        # little-endian y ...
    enc[:, 31] |= (xo[:, 31] & 1) << 7                              # ... with the low bit of x on top
    return t(ok) & (enc == sig[:, :32]).all(dim=1)


def products_per_verification():
    """32x32->64 limb products of one Eddsa::verify (eddsa_sm100.cuh) and of one k_ecnmul2<F_X25519, Edwards> row,
    from the operation counts of the code: M = 64 (8x8 words), S = 36; Montgomery import / export on the order field
    are one product each; dbl = 3M + 4S, add = 11M + S (multiplication by d counted as M)."""
    M, S = 64, 36
    pro = 251 * S + 13 * M                                            # (p-5)/8 chain of 2^255 - 19
    inv = pro + 1 * (S + M) + 3 * S + M                              # Field::inv with PM1D2 = 2
    dbl, add = 3 * M + 4 * S, 11 * M + S
    table = 2 * dbl + 11 * add                                        # 2P, 3P, 2Q, 3Q, nine sums a P + b Q
    loop = 128 * (2 * dbl + add)
    order = 3 * M + M + M                                             # S, h_lo, h_hi imported; h_hi R^2; k exported
    decode = 3 * S + 5 * M + pro + M + (S + M) + M + 2 * M            # u v v^3 u v^3 v^7 u v^7, chain, x, v x^2, sqrt(-1), tighten
    fused = order + decode + M + table + loop + inv + 2 * M           # + negate A; encode: inversion, x, y
    ecnmul2 = 2 * (2 * S + 4 * M) + table + loop + inv + 2 * M        # set x2 (on-curve check, tighten), get
    return fused, ecnmul2


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    parts = [p.strip() for p in q.stdout.strip().splitlines()[0].split(",")] if q.returncode == 0 and q.stdout.strip() else []
    return {"name": parts[0] if parts else None, "power_limit": parts[1] if len(parts) > 1 else None,
            "max_sm_clock": parts[2] if len(parts) > 2 else None}


def signatures(count, seed=5):
    """count (h, sig, pk) byte rows signed by OpenSSL with eight keys."""
    import hashlib
    import random
    from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey
    from cryptography.hazmat.primitives.serialization import Encoding, PublicFormat
    rng = random.Random(seed)
    keys = [Ed25519PrivateKey.from_private_bytes(rng.randbytes(32)) for _ in range(8)]
    pubs = [k.public_key().public_bytes(Encoding.Raw, PublicFormat.Raw) for k in keys]
    out = []
    for i in range(count):
        msg = rng.randbytes(32)
        sig = keys[i % 8].sign(msg)
        out.append((hashlib.sha512(sig[:32] + pubs[i % 8] + msg).digest(), sig, pubs[i % 8]))
    return out


def cpu_baseline(seconds=2.0):
    """OpenSSL (through cryptography) verifications per second on all host cores, one process per core."""
    import multiprocessing as mp
    nproc = os.cpu_count() or 1
    with mp.get_context("spawn").Pool(nproc) as pool:
        counts = pool.map(_cpu_worker, [seconds] * nproc)
    return {"verifications_per_s": sum(counts) / seconds, "processes": nproc,
            "what": "OpenSSL Ed25519 verify through python cryptography (hashing included), one process per host core"}


def _cpu_worker(seconds):
    from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PrivateKey
    k = Ed25519PrivateKey.generate()
    msg = b"x" * 32
    sig = k.sign(msg)
    pk = k.public_key()
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        for _ in range(100):
            pk.verify(sig, msg)
        n += 100
    return n


def timed(fn, min_seconds=1.0):
    """Seconds per call with CUDA events."""
    import torch
    fn()
    torch.cuda.synchronize()
    reps = 1
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


def timed_host(fn, min_seconds=1.0):
    """Seconds per call with the host clock around calls that end in a synchronise (for arms with host work)."""
    import torch
    fn()
    torch.cuda.synchronize()
    reps, total = 0, 0.0
    while total < min_seconds:
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        total += time.perf_counter() - t0
        reps += 1
    return total / reps, reps


def main():
    import numpy as np
    import torch
    from modarith_b200 import lib as mlib
    from modarith_b200.ecn import ecnmul2
    from modarith_b200.eddsa import verify_digest
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
    prods, prods2 = products_per_verification()
    res["products_per_verification"] = prods
    res["products_per_ecnmul2_row"] = prods2
    res["imad_peak_products_per_s"] = peak
    base = signatures(1 << 14)
    cols = [np.frombuffer(b"".join(col), dtype=np.uint8).reshape(len(base), -1) for col in zip(*base)]
    res["rows"] = {}
    for lg in (18, 20, 22):
        n = 1 << lg
        idx = np.arange(n) % len(base)
        h, sig, pk = (torch.from_numpy(np.ascontiguousarray(c[idx])).to(dev) for c in cols)
        bad = torch.from_numpy(np.arange(n) % 4 == 3).to(dev)       # every fourth row: digest changed, must fail
        h[:, 0] ^= bad.to(torch.uint8)
        want = ~bad
        e, f = sig[:, 32:].flip(1).contiguous(), h[:, :32].contiguous()   # ecnmul2 alone: any scalars do
        gx = torch.from_numpy(np.tile(np.frombuffer(GX.to_bytes(32, "big"), dtype=np.uint8), (n, 1))).to(dev)
        gy = torch.from_numpy(np.tile(np.frombuffer(GY.to_bytes(32, "big"), dtype=np.uint8), (n, 1))).to(dev)
        row = {}
        assert torch.equal(verify_digest(h, sig, pk), want), "fused: wrong flags"
        assert torch.equal(composed(h, sig, pk), want), "composed: wrong flags"
        for name, fn, clock in (("fused", lambda: verify_digest(h, sig, pk), timed),
                                ("composed", lambda: composed(h, sig, pk), timed_host),
                                ("ecnmul2", lambda: ecnmul2("ED25519", e, gx, gy, f, gx, gy), timed)):
            t, reps = clock(fn)
            row[name] = {"seconds_per_call": t, "reps": reps, "M_per_s": n / t / 1e6}
        row["fused"]["imad_fraction"] = n * prods / row["fused"]["seconds_per_call"] / peak
        row["ecnmul2"]["imad_fraction"] = n * prods2 / row["ecnmul2"]["seconds_per_call"] / peak
        res["rows"][str(n)] = row
        print(lg, json.dumps(row), flush=True)
        del h, sig, pk, bad, want, e, f, gx, gy
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
