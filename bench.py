#!/usr/bin/env python3
"""bench.py -- X25519 scalar-mults/s on N B200s (BASELINE.json metric), with the INT32-IMAD
roofline, the end-to-end (host buffers, C ABI) figure and the reference's CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--keys 1048576] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (rfc7748: clamp, import, 255 ladder steps, inversion,
export) over one batch of 2^20 random raw key/point pairs per GPU (BASELINE configs[1]).
N>1 is launched by torchrun, one rank per GPU; every rank owns a contiguous key range of the
global batch (weak scaling: 2^20 keys per GPU) and there is NO collective on the data path;
the optional NCCL all-gather of the result strings is timed separately (`gather_ms`).

Printed JSON (rank 0, one line):
  value      keys/s over all GPUs, inputs resident in HBM, CUDA events, max over ranks
  e2e        same metric through mab_X25519_rfc7748_host with pinned HOST buffers (H2D + D2H inside)
  roofline   achieved limb products/s of the ladder kernel vs the IMAD peak measured live by
             the in-library microbenchmark (mab_imad_peak); HBM GB/s shown to be non-binding
  cpu_baseline  the reference's own generated 64-bit C (oracle/_ref) on all host cores, bounded sample
`--impl reference` times only that CPU implementation (rank 0) and prints the same line shape.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NB = 32
CURVE = "X25519"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--keys", type=int, default=1 << 20, help="keys per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="keys in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the X448 / P-256 side measurements")
    ap.add_argument("--single-process", action="store_true",
                    help="N GPUs from ONE process: device-resident launches on every device, and the end-to-end "
                         "figure through mab_X25519_rfc7748_host_multi (one host thread per GPU inside the library)")
    ap.add_argument("--parity-keys", type=int, default=-1,
                    help="keys of EVERY rank's first step checked against the reference build before timing "
                         "(-1 = all local keys, capped at 2^20 per rank)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the X25519 results of the last one to DIR/x25519_out.npy "
                         "([rows, 32] byte values as float32; every key up to 2^18, beyond that a fixed seeded sample "
                         "of 2^18 keys, see dump_rows); with several GPUs, an equal seeded sample of every GPU's "
                         "keys, in key order")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; --impl reference has none")
    return args


# ------------------------------------------------------------------------------------------
def workload_config(n_local, world):
    """The `config` object of the JSON line; both arms print exactly this for the same --gpus / --keys, so that the
    driver's comparison of the two lines sees one workload (what differs between the arms -- the CPU sample of each
    reference step -- is said in `cpu_baseline.sample`)."""
    nsets = 3 if n_local * 3 * 32 <= (1 << 30) else 1
    return {"workload": "batched X25519 (rfc7748) 2^20 random scalars/points per GPU" if n_local == 1 << 20
            else "batched X25519 (rfc7748) %d random scalars/points per GPU" % n_local,
            "keys_per_gpu": n_local, "keys_total": n_local * world, "sharding": "contiguous key ranges, no collective",
            "l2": ("inputs rotate over 3 buffer sets (288 MB > 126 MB L2); kernel moves 96 B/key" if nsets == 3 else
                   "one buffer set of %d MB (>> 126 MB L2); kernel moves 96 B/key" % (n_local * 3 * 32 >> 20)),
            "inputs": "numpy PCG64(7748+...) raw bytes, unclamped / unreduced"}


def make_inputs(n, seed):
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, 256, (n, NB), dtype=np.uint8), rng.integers(0, 256, (n, NB), dtype=np.uint8)


DUMP_ROWS = 1 << 18          # 2^18 keys x 32 bytes as float32 = 32 MiB


def dump_rows(n, m=DUMP_ROWS):
    """Rows of an n-key shard that --dump-outputs writes: all of them up to m, else a fixed seeded sample of m in
    ascending order, so that two builds run with the same arguments write the same rows."""
    import numpy as np
    if n <= m:
        return np.arange(n)
    return np.sort(np.random.Generator(np.random.PCG64(2020)).choice(n, m, replace=False))


def dump_part(out, shards):
    """The rows of one GPU's [n, 32] uint8 result that --dump-outputs writes when `shards` GPUs share the batch."""
    import torch
    return out[torch.from_numpy(dump_rows(out.shape[0], DUMP_ROWS // shards)).to(out.device)]


def dump_outputs(path, parts):
    """parts: dump_part of every GPU's result of the last timed step, in key order."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "x25519_out.npy"), np.concatenate([p.cpu().numpy() for p in parts]).astype(np.float32))


def load_reference():
    """The reference's own C for this path (oracle/_ref/libref_X25519.so).  This is one of the two
    places bench.py may execute oracle/ code: as the CPU baseline, never as the thing shipped."""
    p = os.path.join(ROOT, "oracle", "_ref", "libref_%s.so" % CURVE)
    if not os.path.exists(p):
        return None
    lib = ctypes.CDLL(p)
    lib.ref_max_threads.restype = ctypes.c_int
    return lib


def time_reference(lib, k, u, threads):
    import numpy as np
    out = np.zeros_like(k)
    t0 = time.perf_counter()
    lib.ref_rfc7748_batch(k.ctypes.data_as(ctypes.c_char_p), u.ctypes.data_as(ctypes.c_char_p),
                          out.ctypes.data_as(ctypes.c_char_p), ctypes.c_size_t(k.shape[0]), ctypes.c_int(threads))
    return time.perf_counter() - t0, out


def cpu_baseline_port(sample_keys):
    """Fallback when oracle/_ref has not been built: the plain-C restatement oracle/oracle.c."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    n = sample_keys if sample_keys > 0 else 2048
    k, u = make_inputs(n, 7748)
    c_oracle.rfc7748_batch(CURVE, k[:64], u[:64])
    t0 = time.perf_counter()
    c_oracle.rfc7748_batch(CURVE, k, u)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "scalar-mults/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": "first %d of the 2^20 PCG64(7748) raw key/point pairs; oracle/oracle.c (generic schoolbook "
                      "restatement, OpenMP over all cores) -- oracle/_ref was not available" % n}


def cpu_baseline(sample_keys):
    lib = load_reference()
    if lib is None:
        return cpu_baseline_port(sample_keys)
    cores = os.cpu_count() or 1
    k, u = make_inputs(4096 if sample_keys <= 0 else min(4096, sample_keys), 1)
    time_reference(lib, k, u, cores)                      # warm-up: thread pool, page faults
    dt, _ = time_reference(lib, k, u, cores)              # rate estimate
    rate = k.shape[0] / dt
    n = sample_keys if sample_keys > 0 else 0
    if n == 0:
        n = int(max(1 << 17, min(1 << 20, rate * 1.5)))   # ~1.5 s wall on all cores (about 25-50 CPU-seconds)
    k, u = make_inputs(n, 7748)
    dt, _ = time_reference(lib, k, u, cores)
    return {"value": n / dt, "unit": "scalar-mults/s", "cores": cores, "kind": "reference",
            "per_core": n / dt / cores,
            "sample": "first %d of the 2^20 PCG64(7748) raw key/point pairs; reference's generated 64-bit C "
                      "(pseudo.py 64 X25519 + rfc7748.c, gcc -O3 -march=x86-64-v3, OpenMP over all cores; "
                      "addition chain from the repo's stand-in, not the real addchain)" % n}


class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, t_begin=None, t_end=None, more=()):
        """Summarise the samples whose timestamp falls inside [t_begin, t_end] or one of the `more` windows
        (time.time() values bracketing the timed regions; the sampler itself is started before the warm-up)."""
        if self.proc is None:
            return None
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            try:
                self.proc.kill()
            except Exception:
                pass
        self.f.close()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        import datetime
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            if t_begin is not None:
                try:
                    ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    continue
                if not any(a - 0.02 <= ts <= b + 0.02 for a, b in ((t_begin, t_end),) + tuple(more)):
                    continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


def imad_peak(lib, sms):
    """Measured INT32 multiplier peak in 32x32->64 limb products/s (SURVEY.md 8d).  A product is one
    IMAD.WIDE.U32 or an IMAD.LO+IMAD.HI pair, whichever the chip does faster."""
    res = {}
    blocks, threads, iters = sms * 8, 256, 4000
    for variant, name in ((0, "imad_wide"), (1, "imad_lo"), (2, "imad_hi"), (3, "imad_wide_x_chain"),
                          (4, "wide_plus_1alu"), (5, "wide_plus_2alu"), (6, "iadd3")):
        ms, ins = ctypes.c_float(), ctypes.c_double()
        rc = lib.mab_imad_peak(variant, iters, blocks, threads, ctypes.byref(ms), ctypes.byref(ins), None)
        if rc != 0:
            return None
        res[name] = ins.value / (ms.value * 1e-3)          # thread-level instructions per second
    peak = max(res["imad_wide"], min(res["imad_lo"], res["imad_hi"]) / 2.0, res["imad_wide_x_chain"])
    res["peak_products_per_s"] = peak
    return res


def _time(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def extra_measurements(lib, mlib, dev, peak, hbm_peak):
    """Side figures for the other BASELINE configs (rank 0, one GPU): X448 ladder, P-256 field ops.
    Single field operations per launch are HBM-bound (96 B per 64 products) and reported against the
    measured copy bandwidth; register-resident chains are reported against the IMAD peak."""
    import torch
    from modarith_b200 import Field
    from modarith_b200.rfc7748 import rfc7748
    pk = peak["peak_products_per_s"] if peak else None
    out = {}
    gen = torch.Generator(device=dev).manual_seed(448)
    n = 1 << 20
    k = torch.randint(0, 256, (n, 56), dtype=torch.uint8, device=dev, generator=gen)
    u = torch.randint(0, 256, (n, 56), dtype=torch.uint8, device=dev, generator=gen)
    v = torch.empty_like(k)
    t = _time(lambda: rfc7748("X448", k, u, v), 3)
    prod = mlib.products("X448", "rfc7748")
    out["x448"] = {"workload": "X448 ladder, 2^20 keys", "value": n / t, "unit": "scalar-mults/s",
                   "products_per_key": prod, "imad_frac": (n / t * prod / pk) if pk else None}
    del k, u, v
    # P-256 scalar multiplication (SURVEY.md 8f row 1): ecnXXXset + ecnXXXmul + ecnXXXget, 2^18 points
    try:
        from modarith_b200.ecn import ecnmul
        from modarith_b200.primes import NIST256 as P256
        ne = 1 << 18
        e = torch.randint(0, 256, (ne, 32), dtype=torch.uint8, device=dev, generator=gen)
        import numpy as np
        gx = torch.from_numpy(np.tile(np.frombuffer(P256.wgx.to_bytes(32, "big"), dtype=np.uint8), (ne, 1))).to(dev)
        gy = torch.from_numpy(np.tile(np.frombuffer(P256.wgy.to_bytes(32, "big"), dtype=np.uint8), (ne, 1))).to(dev)
        t = _time(lambda: ecnmul("NIST256", e, gx, gy), 2)
        # algorithmic work of the reference's own schedule (weierstrass.c:494-542): 4 dbl + 3 add for the table,
        # 64 x (4 dbl + 1 add); dbl = 10M + 3S, add = 14M (multiplications by b counted as M), one inversion + 2M
        M, S = 64, 36
        work = (4 + 256) * (10 * M + 3 * S) + (3 + 64) * 14 * M + mlib.products("NIST256", "modinv") + 2 * M
        out["nist256_ecnmul"] = {"workload": "P-256 scalar multiplication (set+mul+get), 2^18 points", "value": ne / t,
                                 "unit": "scalar-mults/s", "products_per_point": work,
                                 "imad_frac": (ne / t * work / pk) if pk else None,
                                 "note": "products_per_point is the REFERENCE's schedule (complete doublings, weierstrass.c:494-542); "
                                         "this build runs the four doublings between digits in Jacobian coordinates (36 products "
                                         "instead of 52 per digit), so like the shared inversions it executes fewer products than "
                                         "the numerator credits"}
        # e*P + f*Q (ecnXXXmul2): this build does one doubling and one addition for each of the 263 joint digits
        from modarith_b200.ecn import ecnmul2
        n2 = ne // 2
        f2 = torch.randint(0, 256, (n2, 32), dtype=torch.uint8, device=dev, generator=gen)
        t = _time(lambda: ecnmul2("NIST256", e[:n2], gx[:n2], gy[:n2], f2, gx[:n2], gy[:n2]), 2)
        work2 = 263 * (10 * M + 3 * S + 14 * M) + 2 * 14 * M + mlib.products("NIST256", "modinv") + 2 * M
        out["nist256_ecnmul2"] = {"workload": "P-256 e*P + f*Q (set x2 + mul2 + get), 2^17 pairs", "value": n2 / t,
                                  "unit": "double-mults/s", "products_per_pair": work2,
                                  "imad_frac": (n2 / t * work2 / pk) if pk else None,
                                  "note": "products_per_pair counts one doubling and one addition for each of the 263 joint digits "
                                          "(round 1's constant-work form of the reference's schedule); this build uses joint 2-bit "
                                          "windows (256 doublings + 141 additions) and executes about 35 % fewer products"}
        # Ed25519 (edwards.c): dbl = 3M + 4S, add = 11M + 1S (multiplication by d counted as M)
        from modarith_b200.primes import X25519 as P255
        gx = torch.from_numpy(np.tile(np.frombuffer(P255.ed_gx.to_bytes(32, "big"), dtype=np.uint8), (ne, 1))).to(dev)
        gy = torch.from_numpy(np.tile(np.frombuffer(P255.ed_gy.to_bytes(32, "big"), dtype=np.uint8), (ne, 1))).to(dev)
        t = _time(lambda: ecnmul("ED25519", e, gx, gy), 2)
        work = (4 + 256) * (3 * M + 4 * S) + (3 + 64) * (11 * M + S) + mlib.products("X25519", "modinv") + 2 * M
        out["ed25519_ecnmul"] = {"workload": "Ed25519 scalar multiplication (set+mul+get), 2^18 points", "value": ne / t,
                                 "unit": "scalar-mults/s", "products_per_point": work,
                                 "imad_frac": (ne / t * work / pk) if pk else None}
        t = _time(lambda: ecnmul2("ED25519", e[:n2], gx[:n2], gy[:n2], f2, gx[:n2], gy[:n2]), 2)
        work2 = 263 * (3 * M + 4 * S + 11 * M + S) + 2 * (11 * M + S) + mlib.products("X25519", "modinv") + 2 * M
        out["ed25519_ecnmul2"] = {"workload": "Ed25519 e*P + f*Q (set x2 + mul2 + get), 2^17 pairs", "value": n2 / t,
                                  "unit": "double-mults/s", "products_per_pair": work2,
                                  "imad_frac": (n2 / t * work2 / pk) if pk else None}
        del e, gx, gy, f2
    except Exception as ex:           # the side measurement must never sink the headline line
        out["nist256_ecnmul"] = {"error": str(ex)[:200]}
    for name, nel in (("NIST256", 1 << 24), ("X25519", 1 << 22)):
        F = Field(name, dev)
        a8 = torch.randint(0, 256, (nel, F.Nbytes), dtype=torch.uint8, device=dev, generator=gen)
        b8 = torch.randint(0, 256, (nel, F.Nbytes), dtype=torch.uint8, device=dev, generator=gen)
        x, _ = F.modimp(a8)
        y, _ = F.modimp(b8)
        del a8, b8
        r = F.alloc(nel)
        L = F.Nlimbs
        res = {"elements": nel}
        t = _time(lambda: F.modmul(x, y, r), 5)
        res["modmul_single_launch"] = {"value": nel / t / 1e9, "unit": "Gop/s", "hbm_GBps": nel * 12 * L / t / 1e9,
                                       "hbm_frac": nel * 12 * L / t / 1e9 / hbm_peak,
                                       "imad_frac": (nel / t * L * L / pk) if pk else None}
        t = _time(lambda: F.modadd(x, y, r), 5)
        res["modadd_single_launch"] = {"value": nel / t / 1e9, "unit": "Gop/s", "hbm_GBps": nel * 12 * L / t / 1e9,
                                       "hbm_frac": nel * 12 * L / t / 1e9 / hbm_peak}
        m, iters = 1 << 21, 512
        xs, ys, rs = x[:, :m].contiguous(), y[:, :m].contiguous(), r[:, :m].contiguous()
        t = _time(lambda: F.bench_modmul(xs, ys, rs, iters), 2)
        res["modmul_register_resident"] = {"value": m * iters / t / 1e9, "unit": "Gop/s", "chain": iters,
                                           "imad_frac": (m * iters / t * L * L / pk) if pk else None}
        t = _time(lambda: F.modnsqr(rs, iters), 2)
        res["modsqr_register_resident"] = {"value": m * iters / t / 1e9, "unit": "Gop/s", "chain": iters,
                                           "imad_frac": (m * iters / t * (L * (L + 1) // 2) / pk) if pk else None}
        pi = mlib.products(name, "modinv")
        t = _time(lambda: F.modinv_perelement(xs, rs), 2)
        res["modinv_one_chain_per_element"] = {"value": m / t / 1e6, "unit": "Mop/s", "products": pi,
                                               "imad_frac": (m / t * pi / pk) if pk else None}
        t = _time(lambda: F.modinv(xs, None, rs), 2)
        res["modinv"] = {"value": m / t / 1e6, "unit": "Mop/s", "products": pi,
                         "imad_frac_reference_work": (m / t * pi / pk) if pk else None,
                         "note": "one progenitor chain shared by 8 elements per thread (Montgomery's trick): executes "
                                 "about 1/6 of the reference algorithm's products, so this fraction can exceed 1"}
        t = _time(lambda: F.modsqrt(xs, None, rs), 2)
        ps = mlib.products(name, "modsqrt")
        res["modsqrt"] = {"value": m / t / 1e6, "unit": "Mop/s", "products": ps, "imad_frac": (m / t * ps / pk) if pk else None}
        if name == "X25519":
            # the reference's own WL=32 limb plan (radix 2^29 x 9, csrc/mab_unsat29.cuh) on the same chain
            ua = torch.randint(0, 1 << 29, (9, m), dtype=torch.int32, device=dev, generator=gen)
            ub = torch.randint(0, 1 << 29, (9, m), dtype=torch.int32, device=dev, generator=gen)
            uc = torch.empty_like(ua)
            st = torch.cuda.current_stream(dev).cuda_stream
            t = _time(lambda: mlib.check(lib.mab_probe_unsat29_modmul(ua.data_ptr(), ub.data_ptr(), uc.data_ptr(),
                                                                      iters, m, m, st)), 2)
            res["modmul_register_resident_unsaturated_9x29"] = {
                "value": m * iters / t / 1e9, "unit": "Gop/s", "chain": iters,
                "imad_frac": (m * iters / t * L * L / pk) if pk else None,
                "note": "comparison kernel on the reference's radix-2^29 x 9 limb plan; same algorithmic 64 products"}
            del ua, ub, uc
        out[name] = res
        del x, y, r, xs, ys, rs
    # a consumer-shaped sequence of field calls (the complete P-256 point addition of weierstrass.c:69-160: 12 modmul +
    # 2 by the curve constant + 29 modadd/modsub) as ONE mab_NIST256_modprog launch against one launch per call
    try:
        F = Field("NIST256", dev)
        m = 1 << 21
        ops = [F.modimp(torch.randint(0, 256, (m, 32), dtype=torch.uint8, device=dev, generator=gen))[0] for _ in range(7)]
        X1_, Y1_, Z1_, X2_, Y2_, Z2_, B_, t0, t1, t2, t3, t4, X3, Y3, Z3 = range(15)
        code = [("mul", t0, X1_, X2_), ("mul", t1, Y1_, Y2_), ("mul", t2, Z1_, Z2_), ("add", t3, X1_, Y1_), ("add", t4, X2_, Y2_),
                ("mul", t3, t3, t4), ("add", t4, t0, t1), ("sub", t3, t3, t4), ("add", t4, Y1_, Z1_), ("add", X3, Y2_, Z2_),
                ("mul", t4, t4, X3), ("add", X3, t1, t2), ("sub", t4, t4, X3), ("add", X3, X1_, Z1_), ("add", Y3, X2_, Z2_),
                ("mul", X3, X3, Y3), ("add", Y3, t0, t2), ("sub", Y3, X3, Y3), ("mul", Z3, B_, t2), ("sub", X3, Y3, Z3),
                ("add", Z3, X3, X3), ("add", X3, X3, Z3), ("sub", Z3, t1, X3), ("add", X3, t1, X3), ("mul", Y3, B_, Y3),
                ("add", t1, t2, t2), ("add", t2, t1, t2), ("sub", Y3, Y3, t2), ("sub", Y3, Y3, t0), ("add", t1, Y3, Y3),
                ("add", Y3, t1, Y3), ("add", t1, t0, t0), ("add", t0, t1, t0), ("sub", t0, t0, t2), ("mul", t1, t4, Y3),
                ("mul", t2, t0, Y3), ("mul", Y3, X3, Z3), ("add", Y3, Y3, t2), ("mul", X3, t3, X3), ("sub", X3, X3, t1),
                ("mul", Z3, t4, Z3), ("mul", t1, t3, t0), ("add", Z3, Z3, t1)]
        outs = [F.alloc(m) for _ in range(3)]
        t = _time(lambda: F.modprog(code, ops, [X3, Y3, Z3], outputs=outs), 3)
        try:
            outs_j = [F.alloc(m) for _ in range(3)]
            F.modprog(code, ops, [X3, Y3, Z3], outputs=outs_j, jit=True)           # compiles (about a second), then cached
            tj = _time(lambda: F.modprog(code, ops, [X3, Y3, Z3], outputs=outs_j, jit=True), 3)
            same = all(bool(torch.equal(a, b)) for a, b in zip(outs, outs_j))
            del outs_j
        except Exception as ex:
            tj, same = None, str(ex)[:200]
        R = [F.alloc(m) for _ in range(15)]
        for k in range(7):
            R[k].copy_(ops[k])

        def separately():
            for op, d, a, b in code:
                (F.modmul if op == "mul" else F.modadd if op == "add" else F.modsub)(R[a], R[b], R[d])
        ts = _time(separately, 2)
        nmul = sum(1 for c in code if c[0] == "mul")
        out["nist256_modprog_point_addition"] = {
            "workload": "complete P-256 point addition as a 43-instruction modprog program, 2^21 point pairs",
            "value": m / t, "unit": "additions/s", "one_launch_per_call_value": m / ts, "speedup": ts / t,
            "field_ops_per_s": m * len(code) / t, "imad_frac": (m / t * nmul * 64 / pk) if pk else None,
            "hbm_bytes_per_addition": 10 * 32, "one_launch_per_call_hbm_bytes": len(code) * 96,
            "compiled": {"note": "mab_NIST256_modprog_jit: the same program compiled by NVRTC, variables in machine registers",
                         "value": (m / tj) if tj else None, "unit": "additions/s",
                         "imad_frac": (m / tj * nmul * 64 / pk) if (tj and pk) else None,
                         "speedup_over_one_launch_per_call": (ts / tj) if tj else None,
                         "identical_to_interpreted": same}}
        del ops, outs, R
    except Exception as ex:
        out["nist256_modprog_point_addition"] = {"error": str(ex)[:200]}
    # the generator's fall-back plan (any odd modulus: full Montgomery with real multiplies), SURVEY.md 8f row 2
    for name in ("SECP256K1", "NIST256ORDER"):
        try:
            F = Field(name, dev)
            m, iters = 1 << 20, 256
            x, _ = F.modimp(torch.randint(0, 256, (m, F.Nbytes), dtype=torch.uint8, device=dev, generator=gen))
            y, _ = F.modimp(torch.randint(0, 256, (m, F.Nbytes), dtype=torch.uint8, device=dev, generator=gen))
            r = F.alloc(m)
            L = F.Nlimbs
            t = _time(lambda: F.bench_modmul(x, y, r, iters), 2)
            out[name] = {"modmul_register_resident": {"value": m * iters / t / 1e9, "unit": "Gop/s", "chain": iters,
                                                      "imad_frac": (m * iters / t * L * L / pk) if pk else None,
                                                      "note": ("PseudoMersenne33 plan: 2^256 == 2^32 + 977, L^2 + L + 1 wide multiplies per modmul" if name == "SECP256K1"
                                                               else "MontgomeryFull plan: word-serial Montgomery, 2 L^2 wide multiplies + L plain ones per modmul")}}
            del x, y, r
        except Exception as ex:
            out[name] = {"error": str(ex)[:200]}
    return out


# ------------------------------------------------------------------------------------------
def run_reference(args, rank):
    if rank != 0:
        return 0
    lib = load_reference()
    if lib is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_X25519.so not built"}))
        return 0
    cores = os.cpu_count() or 1
    k, u = make_inputs(4096, 1)
    dt, _ = time_reference(lib, k, u, cores)
    rate = k.shape[0] / dt
    total_budget_s = 120.0
    n = int(max(4096, min(args.keys, rate * total_budget_s / max(1, args.steps + args.warmup))))
    k, u = make_inputs(n, 7748)
    for _ in range(args.warmup):
        time_reference(lib, k, u, cores)
    t = 0.0
    for _ in range(args.steps):
        d, _ = time_reference(lib, k, u, cores)
        t += d
    v = n * args.steps / t
    sample = ("each step = first %d of the 2^20 PCG64(7748) raw key/point pairs; the reference's generated 64-bit C "
              "(pseudo.py 64 X25519 pasted into rfc7748.c, generic=False, PSCR=False, gcc -O3 -march=x86-64-v3), "
              "OpenMP over %d host threads" % (n, cores))
    print(json.dumps({
        "impl": "reference", "metric": "X25519 scalar-mults/s", "value": v, "unit": "scalar-mults/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (radix 2^51) on CPU",
        "data": "synthetic",
        "config": workload_config(args.keys, max(1, args.gpus)),
        "cpu_baseline": {"value": v, "unit": "scalar-mults/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": v, "unit": "scalar-mults/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))
    return 0


def run_single_process(args):
    """--gpus N --single-process: the C consumer's view of a multi-GPU box (VERDICT r1 item 6).  One process,
    no torchrun, no NCCL: `value` launches the device-pointer call on every device from this thread (the calls are
    asynchronous) and takes the slowest device's CUDA-event time; `e2e` is one mab_X25519_rfc7748_host_multi call
    per step on pinned host buffers holding all N x keys keys."""
    import numpy as np
    import torch
    from modarith_b200 import lib as mlib
    from modarith_b200.rfc7748 import rfc7748
    lib = mlib.load()
    N = args.gpus
    if torch.cuda.device_count() < N:
        raise SystemExit("--single-process --gpus %d needs %d visible devices" % (N, N))
    n_local, n_total = args.keys, args.keys * N
    NSETS = 3
    hk, hu = [], []
    for s in range(NSETS):
        ks, us = [], []
        for g in range(N):
            k, u = make_inputs(n_local, 7748 + 1000 * s + g)
            ks.append(k); us.append(u)
        hk.append(torch.from_numpy(np.concatenate(ks)).pin_memory())
        hu.append(torch.from_numpy(np.concatenate(us)).pin_memory())
    hv = torch.empty((n_total, NB), dtype=torch.uint8).pin_memory()
    dk = [[hk[s][g * n_local:(g + 1) * n_local].to("cuda:%d" % g) for g in range(N)] for s in range(NSETS)]
    du = [[hu[s][g * n_local:(g + 1) * n_local].to("cuda:%d" % g) for g in range(N)] for s in range(NSETS)]
    dv = [torch.empty_like(dk[0][g]) for g in range(N)]

    def step(s):
        for g in range(N):
            with torch.cuda.device(g):
                rfc7748(CURVE, dk[s % NSETS][g], du[s % NSETS][g], dv[g])

    def sync():
        for g in range(N):
            torch.cuda.synchronize(g)

    for w in range(args.warmup):
        step(w)
    sync()
    ev = []
    for g in range(N):
        with torch.cuda.device(g):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ev.append((e0, e1))
    t0 = time.perf_counter()
    for s in range(args.steps):
        step(s)
    for g in range(N):
        with torch.cuda.device(g):
            ev[g][1].record()
    sync()
    wall = time.perf_counter() - t0
    ms = max(e0.elapsed_time(e1) for e0, e1 in ev)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [dump_part(dv[g], N) for g in range(N)])
    # parity of every device's shard against the reference build (set of the last step)
    ref = load_reference()
    parity, pn = None, 0
    if ref is not None:
        s = (args.steps - 1) % NSETS
        m = min(n_local, 1 << 18)
        parity = True
        for g in range(N):
            _, want = time_reference(ref, hk[s][g * n_local:g * n_local + m].numpy(), hu[s][g * n_local:g * n_local + m].numpy(), 0)
            parity = parity and bool(np.array_equal(dv[g][:m].cpu().numpy(), want))
            pn += m
    # end to end through the multi-device C entry point
    fn = lib.mab_X25519_rfc7748_host_multi
    for w in range(2):
        mlib.check(fn(hk[w].data_ptr(), hu[w].data_ptr(), hv.data_ptr(), n_total, N))
    t0 = time.perf_counter()
    for s in range(args.steps):
        mlib.check(fn(hk[s % NSETS].data_ptr(), hu[s % NSETS].data_ptr(), hv.data_ptr(), n_total, N))
    e2e_s = time.perf_counter() - t0
    if ref is not None:
        s = (args.steps - 1) % NSETS
        m = min(n_local, 1 << 18)
        for g in range(N):
            _, want = time_reference(ref, hk[s][g * n_local:g * n_local + m].numpy(), hu[s][g * n_local:g * n_local + m].numpy(), 0)
            parity = parity and bool(np.array_equal(hv[g * n_local:g * n_local + m].numpy(), want))
    print(json.dumps({
        "metric": "X25519 scalar-mults/s", "value": n_total * args.steps / (ms * 1e-3), "unit": "scalar-mults/s",
        "n_gpus": N, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (saturated radix 2^32)", "data": "synthetic",
        "mode": "single-process",
        "config": {"workload": "batched X25519 (rfc7748) %d random scalars/points per GPU" % n_local, "keys_per_gpu": n_local,
                   "keys_total": n_total, "sharding": "contiguous key ranges, one host thread per device inside the library"},
        "wall_ms_per_step": 1e3 * wall / args.steps,
        "e2e": {"value": n_total * args.steps / e2e_s, "unit": "scalar-mults/s", "h2d_bytes_per_step": 2 * NB * n_total,
                "d2h_bytes_per_step": NB * n_total, "ms_per_step": 1e3 * e2e_s / args.steps,
                "api": "mab_X25519_rfc7748_host_multi(bk, bu, bv, n, %d) on pinned host buffers" % N},
        "gpu_launches": args.steps * N, "parity_spot_check": parity, "parity_keys": pn}))
    return 0


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)
    if args.single_process and world == 1 and args.gpus > 1:
        return run_single_process(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from modarith_b200 import lib as mlib
    from modarith_b200.rfc7748 import rfc7748
    from modarith_b200.shard import key_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL announces its version on stdout when the communicator is created; stdout must carry the one JSON
        # line only, so file descriptor 1 points at stderr while the process group comes up
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = mlib.load()
    props = torch.cuda.get_device_properties(dev)
    n_local = args.keys
    n_total = n_local * world
    lo, hi = key_range(rank, world, n_total)
    assert hi - lo == n_local

    # inputs: this rank's contiguous range of the global PCG64(7748) batch; three buffer sets are
    # rotated so no step finds its inputs in L2 (3 x 96 MB > 126 MB)
    NSETS = 3 if n_local * 3 * NB <= (1 << 30) else 1     # one set is already many times L2 beyond 2^23 keys
    hk, hu = [], []
    for s in range(NSETS):
        k, u = make_inputs(n_local, 7748 + 1000 * s + rank)
        hk.append(torch.from_numpy(k).pin_memory())
        hu.append(torch.from_numpy(u).pin_memory())
    dk = [t.to(dev) for t in hk]
    du = [t.to(dev) for t in hu]
    dv = [torch.empty_like(t) for t in dk]
    hv = torch.empty((n_local, NB), dtype=torch.uint8).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity against the reference build before timing: EVERY rank checks its own shard ------
    # (all local keys by default: 2^20 per rank is ~2 s of the reference's C on the host cores, which the
    # ranks share -- each takes cores/world threads)
    ref = load_reference()
    parity = None
    parity_n = 0
    want0 = None
    out0 = rfc7748(CURVE, dk[0], du[0], dv[0])
    torch.cuda.synchronize()
    if ref is not None:
        m = min(n_local, 1 << 20) if args.parity_keys < 0 else min(args.parity_keys, n_local)
        threads = max(1, (os.cpu_count() or 1) // world)
        _, want0 = time_reference(ref, hk[0][:m].numpy(), hu[0][:m].numpy(), threads)
        parity = bool(np.array_equal(out0[:m].cpu().numpy(), want0))
        parity_n = m

    # ---- device-resident throughput --------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                      # running before the warm-up so it is sampling by the timed region
    for w in range(args.warmup):
        rfc7748(CURVE, dk[w % NSETS], du[w % NSETS], dv[w % NSETS])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.time()
    e0.record()
    for s in range(args.steps):
        rfc7748(CURVE, dk[s % NSETS], du[s % NSETS], dv[s % NSETS])
    e1.record()
    barrier()
    t_end = time.time()
    ms = e0.elapsed_time(e1)
    launches = args.steps
    if args.dump_outputs:
        parts = [dump_part(dv[(args.steps - 1) % NSETS], world)]
        if world > 1:
            parts = [torch.empty_like(parts[0]) for _ in range(world)]
            dist.all_gather(parts, dump_part(dv[(args.steps - 1) % NSETS], world))
        if rank == 0:
            dump_outputs(args.dump_outputs, parts)

    # ---- end to end: host buffers through the C ABI (H2D + ladder + D2H inside the timed region) --
    # The buffers are pinned, so the library takes its zero-copy route: one launch whose threads read the
    # keys from host memory and write the results back across PCIe.  The staged three-stream pipeline (what
    # pageable buffers get) is timed beside it for the record.
    def run_e2e(steps):
        for w in range(max(1, min(args.warmup, 2))):
            rfc7748(CURVE, hk[w % NSETS], hu[w % NSETS], hv, device=local)
        barrier()
        t0 = time.perf_counter()
        per = []
        for s in range(steps):
            ts = time.perf_counter()
            rfc7748(CURVE, hk[s % NSETS], hu[s % NSETS], hv, device=local)
            per.append(time.perf_counter() - ts)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, per

    os.environ["MAB_HOST_ZEROCOPY"] = "0"
    staged_s, _ = run_e2e(max(3, args.steps // 2))
    staged_rate = n_local * max(3, args.steps // 2) / staged_s
    os.environ.pop("MAB_HOST_ZEROCOPY")
    t2_begin = time.time()
    e2e_s, e2e_steps = run_e2e(args.steps)
    t2_end = time.time()
    # clocks: samples taken during either timed region (device-resident loop, end-to-end loop); nvidia-smi answers
    # every 20-150 ms depending on the box, and ten 20 ms steps alone can see a single sample
    clocks = sampler.stop(t_begin, t_end, more=((t2_begin, t2_end),)) if rank == 0 else None
    e2e_launches = args.steps
    if want0 is not None:
        # the host-buffer route on the same keys (one more call, outside the timed region)
        hv.zero_()
        rfc7748(CURVE, hk[0], hu[0], hv, device=local)
        parity = parity and bool(np.array_equal(hv[:parity_n].numpy(), want0))

    # ---- optional result gather over NVLink, timed apart ----------------------------------------------
    gather_ms = None
    if world > 1:
        bufs = [torch.empty_like(dv[0]) for _ in range(world)]
        dist.all_gather(bufs, dv[0])
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        dist.all_gather(bufs, dv[0])
        g1.record()
        torch.cuda.synchronize()
        gather_ms = g0.elapsed_time(g1)

    # ---- max over ranks --------------------------------------------------------------------------------
    tt = torch.tensor([ms, e2e_s * 1e3, gather_ms or 0.0], dtype=torch.float64, device=dev)
    # parity: AND over ranks (min), keys compared summed over ranks; -1 = no reference build on this rank
    pp = torch.tensor([(-1 if parity is None else int(parity)), parity_n], dtype=torch.int64, device=dev)
    pmin, psum = pp.clone(), pp.clone()
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(psum, op=dist.ReduceOp.SUM)
    ms, e2e_ms, gather_ms_max = (float(x) for x in tt.cpu())
    parity = None if int(pmin[0]) < 0 else bool(int(pmin[0]))
    parity_total = int(psum[1])

    if rank == 0:
        value = n_total * args.steps / (ms * 1e-3)
        e2e = n_total * args.steps / (e2e_ms * 1e-3)
        prod = mlib.products(CURVE, "rfc7748")
        peak = imad_peak(lib, props.multi_processor_count)
        per_gpu = value / world
        achieved = per_gpu * prod
        roof = {"bound": "int32-imad", "achieved": achieved / 1e9, "peak": None, "unit": "Gprod/s", "frac": None,
                "traffic": None,
                "products_per_key": prod,
                "note": "achieved = keys/s/GPU x %d algorithmic 32x32->64 limb products per X25519 scalar-mult "
                        "(255 x (5M+4S+1 mli) + 251S+13M progenitor + inversion wrapper + final M, L=8); peak = "
                        "IMAD-pipe products/s measured live by mab_imad_peak on this GPU.  The kernel shares one "
                        "inversion among up to four keys per thread (Montgomery's trick), so it EXECUTES fewer products "
                        "than this reference-algorithm count (about 9 700 fewer per key where sharing is four-way); the "
                        "numerator is deliberately the reference's work per key, as SURVEY.md 8d defines it" % prod}
        if peak:
            roof["peak"] = peak["peak_products_per_s"] / 1e9
            roof["frac"] = achieved / peak["peak_products_per_s"]
            roof["microbench_Ginstr_per_s"] = {k: v / 1e9 for k, v in peak.items() if k != "peak_products_per_s"}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            hbm_peak, src = peaks["hbm_gbs"], "measured"
        except Exception:
            hbm_peak, src = 6650.0, "fallback"
        hbm_ach = per_gpu * 3 * NB / 1e9
        roof["hbm"] = {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                       "peak_source": src, "note": "96 algorithmic bytes per key: HBM is not binding"}
        tr = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tr):
            try:
                roof["traffic"] = json.load(open(tr)).get("k_rfc7748_X25519_dram_bytes_per_launch")
            except Exception:
                pass
        extra = None if args.no_extra else extra_measurements(lib, mlib, dev, peak, hbm_peak)
        base = None if args.no_cpu_baseline else cpu_baseline(args.cpu_sample)
        line = {
            "metric": "X25519 scalar-mults/s", "value": value, "unit": "scalar-mults/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (saturated radix 2^32)",
            "data": "synthetic",
            "config": workload_config(n_local, world),
            "e2e": {"value": e2e, "unit": "scalar-mults/s", "h2d_bytes_per_step": 2 * NB * n_local,
                    "d2h_bytes_per_step": NB * n_local, "ms_per_step": e2e_ms / args.steps,
                    "ms_per_step_min_median_max_rank0": [1e3 * min(e2e_steps), 1e3 * statistics.median(e2e_steps),
                                                         1e3 * max(e2e_steps)],
                    "api": "mab_X25519_rfc7748_host on pinned host buffers: one launch, the kernel reads the keys and "
                           "writes the results across PCIe itself (zero-copy); pageable buffers take the staged pipeline",
                    "staged_pipeline_value_rank0": staged_rate},
            "gpu_launches": launches, "gpu_launches_e2e": e2e_launches,
            "roofline": roof, "cpu_baseline": base, "clocks": clocks, "parity_spot_check": parity,
            "parity_keys": parity_total, "parity_ranks": world,
            "parity_note": "every rank compared its own keys (device-pointer call and host-buffer call) byte-for-byte "
                           "with the reference's generated C; parity_spot_check = AND over ranks, parity_keys = sum",
            "gather_ms": gather_ms_max if world > 1 else None, "gpu": props.name, "sms": props.multi_processor_count,
            "extra": extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
