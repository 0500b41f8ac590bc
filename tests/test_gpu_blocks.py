"""Every generated field block on sm_100a at the edges of its representation, word for word against the generator's
interpreter.

Every kernel relies on the bound invariants of the limb plans (gen/plan.py, DESIGN section 2): stored values stay below
`plan.bound`; on the plans with a spare bit, products stay below `plan.tight`, which add_tt / sub_tt assume; mul_w /
sqr_w stay below R inside modpro / modnsqr chains; canon is right over the whole raw range below 2^(32L).
`Plan.self_check` proves them on the interpreter (`Asm.run`) only.  Here a small probe (tests/gpuprobe/blocks.cu),
compiled for every named modulus, runs each block on the device with planted stored words: 0, 1, 2, p-2 .. p+1,
2p-1 .. 2p+1, the top of the block's operand domain minus 1, 2, 2^32, 2^224 and 2^(n-1), 2^n - 1, 2^n, 2^n + c, the
fold constants, runs of all-ones words from either end, alternating words, single bits, the edges of
`Plan.sample_values` and, for the tight bound, those of self_check.  Binary blocks take the full edge x edge cross
product, every block 2^14 sampled values on top.  Each row is checked

  * for its value mod p (R^-1 applied on the Montgomery plans) and canon's flag,
  * for the block's output bound,
  * against the interpreter, word for word (the device code is the interpreter's own instruction sequence), on the
    edge rows and 1024 sampled ones,
  * on the built-in moduli, against the host simulation (tests/hostsim) on every row.

The same planted words then go through the public entry points, and the ladders through saturated word patterns.
Without a GPU the probe is still compiled for every modulus, and the interpreter is checked against the host
simulation on the edge rows."""
import concurrent.futures as cf
import ctypes
import multiprocessing
import os
import random
import subprocess

import numpy as np
import pytest

import util
from modarith_b200.gen.plan import M32, make_plan, value, words
from modarith_b200.primes import ALL_PRIMES, ORDER_PRIMES, REFERENCE_PRIMES, Prime, named

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
PROBE_SRC = os.path.join(ROOT, "tests", "gpuprobe", "blocks.cu")

# 2^383 - 187 with the Montgomery curve the add-on library of that name is built with (__graft_entry__.build)
M383 = Prime("M383", 2**383 - 187, "monty", a24=516287, cof=3, generator=12)
MODULI = dict(ALL_PRIMES, **ORDER_PRIMES)
MODULI.update((n, named(n)) for n in REFERENCE_PRIMES)
MODULI["M383"] = M383
BUILTIN = list(ALL_PRIMES)
ADDONS = ["NIST384", "ED248", "C41417", "NIST521", "M383"]          # the add-on libraries __graft_entry__.build() makes

# same order as ProbeOp in tests/gpuprobe/blocks.cu
BLOCKS = ["mul", "sqr", "mli", "mla", "add", "sub", "neg", "canon", "add_tt", "sub_tt", "mul_w", "sqr_w", "nres", "redc"]
BINARY = ("mul", "add", "sub", "add_tt", "sub_tt", "mul_w")
SCALARS = [0, 1, 2, 39081, 121665, (1 << 31) - 1, M32]
NSAMPLE = 1 << 14
NINTERP = 1024                  # sampled rows also run through the interpreter (0.1 - 2 ms a call)
SIM_OP = {"mul": "MUL", "sqr": "SQR", "mli": "MLI", "mla": "MLA", "add": "ADD", "sub": "SUB", "neg": "NEG",
          "canon": "CANON", "add_tt": "ADDTT", "sub_tt": "SUBTT", "mul_w": "MULW", "sqr_w": "SQRW", "nres": "NRES",
          "redc": "REDCW"}

_plans = {}


def _plan(name):
    if name not in _plans:
        _plans[name] = make_plan(MODULI[name])
    return _plans[name]


def _blocks(plan):
    return [b for b in BLOCKS if b in plan.blocks or b in ("nres", "redc")]


def _domain(plan, block):
    """Exclusive bound of the stored words the block accepts."""
    if block in ("add_tt", "sub_tt"):
        return plan.tight
    if block in ("mul_w", "sqr_w"):
        return plan.weak_bound
    if block == "canon" or (block == "nres" and plan.R != 1):
        return 1 << (32 * plan.L)           # raw imports: canon and, on Montgomery plans, nres take any L words
    return plan.bound                       # (nres is a copy on the plain-residue plans: its output is its input)


def _out_bound(plan, block):
    if block in ("mul", "sqr"):
        return plan.tight or plan.bound
    if block in ("mul_w", "sqr_w"):
        return plan.weak_bound
    if block in ("canon", "redc"):
        return plan.p
    return plan.bound


def edges(plan, D):
    """The representation edges below the domain bound D, sorted."""
    p, L, n = plan.p, plan.L, plan.P.nbits
    c = (1 << n) - p
    e = [0, 1, 2, p - 2, p - 1, p, p + 1, 2 * p - 1, 2 * p, 2 * p + 1,
         D - 1, D - 2, D - (1 << 32), D - (1 << 224), D - (1 << (n - 1)), (1 << n) - 1, 1 << n, (1 << n) + c]
    e += [getattr(plan, k) for k in ("c", "fold", "cl", "d") if isinstance(getattr(plan, k, None), int)]
    e += [value([M32] * k + [0] * (L - k)) for k in range(1, L + 1)]
    e += [value([0] * k + [M32] * (L - k)) for k in range(1, L)]
    e += [value([M32 if i % 2 == j else 0 for i in range(L)]) for j in (0, 1)]
    e += [1 << 31, 1 << 32, 1 << (n - 1)]
    e += plan.sample_values(random.Random(0), 0)             # its edge list alone
    if D == plan.tight:                                      # self_check's tight-bound edges (Plan.self_check)
        T, top = plan.tight, 1 << (32 * L - 1)
        e += [37, 38, 39, T - 1, T - 2, T - 38, T - 39, top - 1, top, top + 1, M32, (1 << 32) - 38]
    return sorted({v for v in e if 0 <= v < D})


def _sample(rng, D, L, k):
    """k values below D with Plan.sample_values' mix: uniform, word patterns, just below the bound."""
    out = []
    for _ in range(k):
        r = rng.random()
        if r < 0.6:
            out.append(rng.randrange(D))
        elif r < 0.8:
            out.append(value([rng.choice([0, M32, 1, 0x80000000, rng.getrandbits(32)]) for _ in range(L)]) % D)
        else:
            out.append((D - 1 - rng.getrandbits(rng.randrange(1, 40))) % D)
    return out


def rows(plan, block):
    """Operand lists (a, b, c, s) of one block, the edge rows first, then NSAMPLE sampled ones; and the edge count.
    b is the second operand of the binary blocks, c mla's addend, s the small integer of mli / mla."""
    D = _domain(plan, block)
    E = edges(plan, D)
    rng = random.Random("%s.%s" % (plan.name, block))
    scal = SCALARS + ([plan.P.a24] if plan.P.a24 else [])
    a, b, c, s = [], [], [], []
    if block in BINARY or block == "mla":
        a = [x for x in E for _ in E]
        (c if block == "mla" else b).extend(y for _ in E for y in E)
        if block == "mla":
            s = [scal[i % len(scal)] for i in range(len(a))]
    elif block == "mli":
        a = [x for x in E for _ in scal]
        s = [t for _ in E for t in scal]
    else:
        a = list(E)
    n_edge = len(a)
    a += _sample(rng, D, plan.L, NSAMPLE)
    if block in BINARY:
        b += _sample(rng, D, plan.L, NSAMPLE)
    if block == "mla":
        c += _sample(rng, D, plan.L, NSAMPLE)
    if block in ("mli", "mla"):
        s += [rng.choice(scal) for _ in range(NSAMPLE)]
    n = len(a)
    return a, b or [0] * n, c or [0] * n, s or [0] * n, n_edge


def interpret(plan, block, x, y, z, t):
    """(stored result, canon's flag) of one row on the generator's interpreter."""
    L = plan.L
    if block in ("nres", "redc"):
        if plan.R == 1:
            return (x, 0) if block == "nres" else (plan.run("canon", a=words(x, L))[0], 0)
        k = plan.R2 if block == "nres" else 1
        return plan.run("mul", a=words(x, L), b=words(k, L))[0], 0
    if block == "neg":
        return plan.run("neg", b=words(x, L))[0], 0
    if block == "canon":
        r, e = plan.run("canon", a=words(x, L))
        return r, e["lt"]
    ins = {"a": words(x, L)}
    if block in BINARY:
        ins["b"] = words(y, L)
    if block == "mla":
        ins["c"] = words(z, L)
    if block in ("mli", "mla"):
        ins["b"] = t
    return plan.run(block, **ins)[0], 0


def expected_ok(plan, block, x, y, z, t, r, f):
    """The value and bound checks of one row."""
    p, R = plan.p, plan.R
    Ri = pow(R, -1, p)
    if block == "canon" and R != 1 and x >= 2 * p:
        # a Montgomery plan's canon is one conditional subtraction: raw words at or above 2p only get their flag
        # (Field::import_raw takes the value through nres); the words are still checked against the interpreter
        return f == 0
    if r >= _out_bound(plan, block):
        return False
    if block == "canon":
        return r == x % p and f == int(x < p)
    if block == "redc":
        return r == x * Ri % p
    if block == "nres" and R == 1:
        return r == x
    want = {"mul": x * y * Ri, "mul_w": x * y * Ri, "sqr": x * x * Ri, "sqr_w": x * x * Ri, "mli": x * t,
            "mla": x * t + z, "add": x + y, "add_tt": x + y, "sub": x - y, "sub_tt": x - y, "neg": -x,
            "nres": x * R}[block]
    return r % p == want % p


def _interpret_modulus(name):
    """Interpreter results of every block of one modulus on its edge rows and NINTERP sampled ones (worker process)."""
    plan = _plan(name)
    out = {}
    for block in _blocks(plan):
        a, b, c, s, ne = rows(plan, block)
        out[block] = [interpret(plan, block, *v) for v in list(zip(a, b, c, s))[:ne + NINTERP]]
    return out


# ---- building the probe -----------------------------------------------------------------------------------------------
def _generate(name, path):
    from modarith_b200.gen.cli import generate
    generate(MODULI[name], path, verbose=False)


def _build_probes(d):
    """field_<NAME>.cuh for every modulus (the generator's self_check included) and libprobe_<NAME>.so from it.
    Returns {name: path or the compiler's complaint}."""
    from modarith_b200.build import _nvcc
    gen = os.path.join(d, "gen")
    os.makedirs(gen, exist_ok=True)
    ctx = multiprocessing.get_context("spawn")
    with cf.ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1), mp_context=ctx) as ex:
        list(ex.map(_generate, MODULI, [os.path.join(gen, "field_%s.cuh" % n) for n in MODULI]))
    nvcc = _nvcc()

    def one(name):
        so = os.path.join(d, "libprobe_%s.so" % name)
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
               "-I", gen, "-I", os.path.join(ROOT, "modarith_b200", "csrc"),
               '-DPROBE_HEADER="field_%s.cuh"' % name, "-DPROBE_FIELD=F_%s" % name, PROBE_SRC, "-o", so]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        return so if r.returncode == 0 else "nvcc failed for %s:\n%s" % (name, r.stdout[-4000:])

    with cf.ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        return dict(zip(MODULI, ex.map(one, MODULI)))


@pytest.fixture(scope="module")
def probes(tmp_path_factory):
    return _build_probes(str(tmp_path_factory.mktemp("gpuprobe")))


@pytest.fixture(scope="module")
def interp():
    """Interpreter results per modulus, computed in worker processes while the device tests run."""
    ctx = multiprocessing.get_context("spawn")
    ex = cf.ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1), mp_context=ctx)
    futs = {name: ex.submit(_interpret_modulus, name) for name in sorted(MODULI, key=lambda n: -_plan(n).L)}
    yield futs
    ex.shutdown(cancel_futures=True)


def _load(probes, name):
    path = probes[name]
    assert os.path.exists(path), path
    lib = ctypes.CDLL(path)
    lib.probe_block.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 6 + [ctypes.c_int, ctypes.c_void_p]
    lib.probe_block.restype = ctypes.c_int
    return lib


# ---- limb planes <-> Python integers ------------------------------------------------------------------------------------
def planes_of(vals, L):
    raw = b"".join(v.to_bytes(4 * L, "little") for v in vals)
    return np.frombuffer(raw, dtype=np.uint32).reshape(len(vals), L).T.copy()


def ints_of(planes):
    L, n = planes.shape
    raw = np.ascontiguousarray(planes.view(np.uint32).T).tobytes()
    return [int.from_bytes(raw[4 * L * i:4 * L * (i + 1)], "little") for i in range(n)]


def _dev(vals, L):
    import torch
    return torch.from_numpy(planes_of(vals, L).view(np.int32)).cuda()


def run_probe(lib, plan, block, a, b, c, s):
    """One block on the device: (stored results, flags)."""
    import torch
    L, n = plan.L, len(a)
    A, B, C = _dev(a, L), _dev(b, L), _dev(c, L)
    S = torch.from_numpy(np.array(s, dtype=np.uint32).view(np.int32)).cuda()
    r = torch.empty((L, n), dtype=torch.int32, device="cuda")
    f = torch.empty(n, dtype=torch.int32, device="cuda")
    rc = lib.probe_block(BLOCKS.index(block), A.data_ptr(), B.data_ptr(), C.data_ptr(), S.data_ptr(), r.data_ptr(),
                         f.data_ptr(), n, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, "probe launch failed: cudaError %d" % rc
    return ints_of(r.cpu().numpy()), f.cpu().numpy().tolist()


def _sim_row(S, block, x, y, z, t):
    if block == "mla":
        r, ret, _ = S.raw("MLA", x, z, scalar=t)
    else:
        r, ret, _ = S.raw(SIM_OP[block], x, y if block in BINARY else None, scalar=t)
    return r, (ret if block == "canon" else 0)


def _fmt(block, x, y, z, t):
    return "%s a=%#x b=%#x c=%#x s=%d" % (block, x, y, z, t)


# ---- without a GPU: the probe compiles for every modulus, the interpreter and the host simulation agree ----------------
@pytest.mark.parametrize("name", list(MODULI))
def test_probe_compiles(probes, name):
    """The generated header of every named modulus compiles for sm_100a inside the probe; most of them are compiled
    nowhere else."""
    lib = _load(probes, name)
    assert lib.probe_limbs() == _plan(name).L


def test_edge_sets_reach_the_domain_tops():
    for name in MODULI:
        plan = _plan(name)
        for block in _blocks(plan):
            D = _domain(plan, block)
            E = edges(plan, D)
            assert E[0] == 0 and E[-1] == D - 1 and D - 2 in E, (name, block)
            if D > 2 * plan.p + 1:
                assert {plan.p - 1, plan.p, 2 * plan.p, 2 * plan.p + 1} <= set(E), (name, block)


@pytest.mark.parametrize("name", BUILTIN)
def test_interpreter_matches_host_simulation_on_edges(hostsim, name):
    """The C transcription of every block (gen/ptx.py emit_sim), which the CPU suite uses in place of the device,
    gives the interpreter's words on every edge row; the value and bound checks hold there too."""
    plan, S = _plan(name), util.Sim(hostsim, name)
    for block in _blocks(plan):
        a, b, c, s, ne = rows(plan, block)
        for v in list(zip(a, b, c, s))[:ne]:
            want = interpret(plan, block, *v)
            assert _sim_row(S, block, *v) == want, _fmt(block, *v)
            assert expected_ok(plan, block, *v, *want), _fmt(block, *v)


# ---- on the device -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODULI))
def test_blocks_on_device(probes, interp, hostsim, name):
    plan, lib = _plan(name), _load(probes, name)
    S = util.Sim(hostsim, name) if name in BUILTIN else None
    mine = {}
    for block in _blocks(plan):
        a, b, c, s, ne = rows(plan, block)
        got, flags = run_probe(lib, plan, block, a, b, c, s)
        mine[block] = (got, flags)
        bad = [i for i in range(len(a)) if not expected_ok(plan, block, a[i], b[i], c[i], s[i], got[i], flags[i])]
        assert not bad, "%d rows wrong or out of bound, first: %s" % (len(bad), _fmt(block, a[bad[0]], b[bad[0]], c[bad[0]], s[bad[0]]))
        if S is not None:
            for i in range(len(a)):
                assert (got[i], flags[i] if block == "canon" else 0) == _sim_row(S, block, a[i], b[i], c[i], s[i]), \
                    "host simulation: " + _fmt(block, a[i], b[i], c[i], s[i])
    want = interp[name].result()
    for block, (got, flags) in mine.items():
        a, b, c, s, ne = rows(plan, block)
        for i, (r, f) in enumerate(want[block]):
            assert (got[i], flags[i] if block == "canon" else 0) == (r, f), \
                "interpreter (%s row): %s" % ("edge" if i < ne else "sampled", _fmt(block, a[i], b[i], c[i], s[i]))



# ---- the same planted words through the public entry points ----------------------------------------------------------------
def _oracle(name):
    from field_oracle import FieldOracle
    from oracle_primes import OraclePrime
    return FieldOracle(name if name in BUILTIN else OraclePrime(name, MODULI[name].p))


@pytest.mark.gpu
@pytest.mark.parametrize("name", BUILTIN + ADDONS)
def test_public_entry_points_on_planted_words(probes, name):
    """Stored edge words planted as raw planes: the element-wise entry points give the probe's words, everything gives
    the oracle's values, and one program over the same inputs (interpreted and compiled) gives the separate calls'
    planes."""
    import torch
    from modarith_b200 import Field
    plan, lib, O = _plan(name), _load(probes, name), _oracle(name)
    F, L, p = Field(name), plan.L, plan.p
    E = edges(plan, plan.bound)
    xs, ys = [x for x in E for _ in E], [y for _ in E for y in E]
    X, Y, X1 = _dev(xs, L), _dev(ys, L), _dev(E, L)
    xv, yv, ev = [plan.from_internal(v) for v in xs], [plan.from_internal(v) for v in ys], [plan.from_internal(v) for v in E]
    r, r1 = F.alloc(len(xs)), F.alloc(len(E))

    def words_of(t):
        return ints_of(t.cpu().numpy())

    def probe(block, a, b=None, s=0):
        n = len(a)
        return run_probe(lib, plan, block, a, b or [0] * n, [0] * n, [s] * n)[0]

    F.modmul(X, Y, r)
    assert words_of(r) == probe("mul", xs, ys) and F.to_ints(r) == [O.modmul(a, b) for a, b in zip(xv, yv)]
    F.modadd(X, Y, r)
    assert words_of(r) == probe("add", xs, ys) and F.to_ints(r) == [O.modadd(a, b) for a, b in zip(xv, yv)]
    F.modsub(X, Y, r)
    assert words_of(r) == probe("sub", xs, ys) and F.to_ints(r) == [O.modsub(a, b) for a, b in zip(xv, yv)]
    F.modsqr(X1, r1)
    assert words_of(r1) == probe("sqr", E) and F.to_ints(r1) == [O.modsqr(a) for a in ev]
    F.modneg(X1, r1)
    assert words_of(r1) == probe("neg", E) and F.to_ints(r1) == [O.modneg(a) for a in ev]
    for s in SCALARS[:-1] + ([plan.P.a24] if plan.P.a24 else []):      # modmli takes 0 <= b < 2^31
        F.modmli(X1, s, r1)
        assert words_of(r1) == probe("mli", E, s=s) and F.to_ints(r1) == [O.modmli(a, s) for a in ev], s
    F.redc(X1, r1)
    assert words_of(r1) == probe("redc", E) == ev
    F.nres(X1, r1)
    assert words_of(r1) == probe("nres", E)
    # the rest on values
    F.modcpy(X1, r1); F.modnsqr(r1, 3)
    assert F.to_ints(r1) == [O.modnsqr(a, 3) for a in ev]
    F.modinv(X1, None, r1)
    assert F.to_ints(r1) == [O.modinv(a) for a in ev]
    F.modsqrt(X1, None, r1)
    assert F.to_ints(r1) == [O.modsqrt(a) for a in ev]
    F.modpro(X1, r1)
    assert F.to_ints(r1) == [O.modpro(a) for a in ev]
    assert F.modqr(None, X1).cpu().tolist() == [O.modqr(None, a) for a in ev]
    F.modcpy(X1, r1); F.modhaf(r1)
    assert F.to_ints(r1) == [O.modhaf(a) for a in ev]
    assert F.modcmp(X, Y).cpu().tolist() == [int(a == b) for a, b in zip(xv, yv)]
    assert F.modis0(X1).cpu().tolist() == [int(a == 0) for a in ev]
    assert F.modis1(X1).cpu().tolist() == [int(a == 1) for a in ev]
    assert F.modsign(X1).cpu().tolist() == [a & 1 for a in ev]
    assert F.to_ints(X1) == ev                                            # modexp
    # one program over the planted inputs: the same planes as the separate calls
    code = [("mul", 2, 0, 1), ("sqr", 3, 0, 0), ("add", 4, 0, 1), ("sub", 5, 0, 1), ("neg", 6, 1, 0),
            ("mli", 7, 0, 0, 121665), ("inv", 8, 0, 0)]
    sep = []
    for op in code:
        t = F.alloc(len(xs))
        if op[0] in ("mul", "add", "sub"):
            getattr(F, "mod" + op[0])(X, Y, t)
        elif op[0] == "sqr":
            F.modsqr(X, t)
        elif op[0] == "neg":
            F.modneg(Y, t)
        elif op[0] == "mli":
            F.modmli(X, op[4], t)
        else:
            F.modinv_perelement(X, t)                # the program inverts element by element too
        sep.append(t)
    for jit in (False, True):
        outs = F.modprog(code, [X, Y], [op[1] for op in code], jit=jit)
        for op, got, want in zip(code, outs, sep):
            assert torch.equal(got, want), (name, jit, op)


# ---- ladders on saturated word patterns -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("curve", ["X25519", "X448", "M383"])
def test_ladder_saturated_word_patterns(curve):
    """Scalars and u-coordinates made of all-ones / all-zero / single-bit words (tests/test_hostsim.py's patterns on 4096
    rows), through the default kernel (shared inversion) and the one-key-per-thread kernel: the operands most likely to
    break a bound the ladder step relies on.  X25519 / X448 against the plain-C oracle on every row, M383 against the
    value-level oracle on the planted rows and 1024 others."""
    import torch
    from modarith_b200 import lib as mlib
    from modarith_b200.rfc7748 import rfc7748
    P = MODULI[curve]
    nb, p, n = 4 * ((P.nbits + 31) // 32), P.p, 4096
    rng = np.random.default_rng(255)
    pats = np.array([0x00, 0xff, 0x80, 0x01, 0x7f, 0xfe], dtype=np.uint8)
    k = np.repeat(pats[rng.integers(0, len(pats), (n, nb // 4))], 4, axis=1).astype(np.uint8)
    u = np.repeat(pats[rng.integers(0, len(pats), (n, nb // 4))], 4, axis=1).astype(np.uint8)
    k[:4] = 0xff
    u[:2] = 0xff
    u[2:4] = 0
    planted = [p - 1, p, p + 1, 2 * p - 1, p - 2, (1 << (8 * nb - 1)) - 1, (1 << (8 * nb)) - 1, 1 << P.nbits]
    for i, v in enumerate(planted):
        u[4 + i] = np.frombuffer((v % (1 << (8 * nb))).to_bytes(nb, "little"), dtype=np.uint8)
    head = 4 + len(planted)
    if curve == "M383":
        from field_oracle import rfc7748 as oracle_rfc7748
        from oracle_primes import OraclePrime
        O = OraclePrime("M383", p, a24=P.a24, cof=P.cof, generator=P.generator)
        rows_ = util.sample_rows(n, 1024, head=head)
        want = np.array([np.frombuffer(oracle_rfc7748(O, k[i].tobytes(), u[i].tobytes()), dtype=np.uint8) for i in rows_])
    else:
        import c_oracle
        rows_, want = np.arange(n), c_oracle.rfc7748_batch(curve, k, u)
    dk, du = torch.from_numpy(k).cuda(), torch.from_numpy(u).cuda()
    got = rfc7748(curve, dk, du)
    out = torch.empty_like(dk)
    lib = mlib.load_for(curve)
    mlib.check(getattr(lib, "mab_%s_rfc7748_perkey" % curve)(dk.data_ptr(), du.data_ptr(), out.data_ptr(), n,
                                                              torch.cuda.current_stream().cuda_stream), "perkey", lib)
    for g in (got, out):
        g = g.cpu().numpy()[rows_]
        bad = np.nonzero((g != want).any(axis=1))[0]
        assert not len(bad), (curve, "rows", rows_[bad[:8]].tolist())
