"""Scalar multiplication and signature verification at the exceptional inputs of the group law.

`EcnMul::mul` (fixed window, signed digits), `EcnMul::mul2w` (joint 2-bit windows over T[a + 4b] = aP + bQ), the complete
Weierstrass formulas with their Jacobian doubling runs and the Edwards law meet equal, opposite and infinite operands
only at special inputs, which random scalars on multiples of the generator never reach.  Seeded sets of such inputs:

  * points: the generators, their negatives, a random multiple; on P-256 the two points with x = 0 (also given with
    x = p), the points with the smallest positive x and three rows off the curve; on Ed25519 all eight torsion points,
    B + T for each of them, and the same points with x + p, y + p or y + 2p (modimp semantics);
  * scalars: 0 .. 17, 2^k and 2^k - 1 (every k on the generators), n - 2 .. n + 2 and the multiples of n below 2^256,
    2^256 - 1, 2^256 - n, (n +- 1) / 2, the nibble runs with the longest recoding carry chains, random ones of each
    parity;
  * e*P + f*Q: Q = O (an input off the curve), +-P, +-2P, +-3P and on Ed25519 every torsion point, so that table entries
    coincide or are O and the additions see equal or opposite operands; (e, f) with e*P + f*Q = O, and pairs that
    share their top 2j bits with Q = -P so that the accumulator stays at O for j digits;
  * ECDSA rows whose u1 G + u2 Q has its halves coincide or cancel, built valid by construction, with h + n, s + 1 and
    h + 1 variants; keys with x = p that the strict key check must reject;
  * Ed25519 rows with small-order and mixed-order keys, k = h mod L at its edges, S at its edges, R = enc([S]B - [k]A)
    and R with its sign bit flipped; keys with a non-canonical y that strict decoding must reject.

Every expected value comes from the Python-integer oracles (field_oracle, ecdsa_oracle, eddsa_oracle).  Without a GPU
every row runs through the host simulation (tests/hostsim), which also aborts on any add_tt / sub_tt operand above its
bound.  On the GPU every row runs through the public entry points in one batch per group, then tiled to 2^18 rows in a
seeded permutation (the rows land in other CTAs, persistent-grid passes and workspace table slices), and ecnmul /
ecnmul2 also run through views at byte offsets 1, 4 and 8 (the byte, word and uint2 paths of aos_ld / aos_st)."""
import ctypes
import multiprocessing as mp
import os
import random
import subprocess

import numpy as np
import pytest

import ecdsa_oracle as EO
import eddsa_oracle as DO
import field_oracle

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
M256 = 1 << 256
PRIME = {"NIST256": "NIST256", "ED25519": "X25519"}
CURVES = list(PRIME)
NTILE = 1 << 18
GROUPS = ["ecnmul NIST256", "ecnmul ED25519", "ecnmul2 NIST256", "ecnmul2 ED25519", "ecdsa", "eddsa"]
# distinct rows per group; the sets are seeded, so a change here is a change of the sets
ROWS = {"ecnmul NIST256": 991, "ecnmul ED25519": 1771, "ecnmul2 NIST256": 697, "ecnmul2 ED25519": 1194,
        "ecdsa": 570, "eddsa": 1004}


def be(v):
    assert 0 <= v < M256, hex(v)
    return v.to_bytes(32, "big")


def nib(s):
    return int(s * (64 // len(s)), 16)


# ---- points ---------------------------------------------------------------------------------------------------------------
SQRT_B = pow(EO.B, (EO.P + 1) // 4, EO.P)


def _p256_xmin():
    """The smallest x > 0 of a P-256 point, and its y."""
    p, x = EO.P, 1
    while True:
        v = (x ** 3 - 3 * x + EO.B) % p
        y = pow(v, (p + 1) // 4, p)
        if y * y % p == v:
            return x, y
        x += 1


def _ed_torsion():
    """The eight points of order dividing 8, by name: O, (0, -1), (+-sqrt(-1), 0) and T8, 3 T8, 5 T8, 7 T8."""
    p = DO.P
    t = {"O": DO.IDENTITY, "T2": (0, p - 1), "T4": (DO.SQRT_M1, 0), "-T4": (p - DO.SQRT_M1, 0)}
    y = 2
    while True:                                  # [L] P for a point P of order 8 L is a point of order 8
        x = DO.recover_x(y, 0)
        if x is not None:
            T = DO.mul(DO.L, (x, y))
            if DO.mul(4, T) != DO.IDENTITY:
                break
        y += 1
    for k in (1, 3, 5, 7):
        t["%dT8" % k] = DO.mul(k, T)
    return t


def _order(add, O, P):
    k, Q = 1, P
    while Q != O:
        Q, k = add(Q, P), k + 1
    return k


def points(curve):
    """{name: (x, y)} in three kinds: 'on' (canonical, on the curve), 'noncanon' (a coordinate >= p that reduces to a
    point of the curve) and 'off' (not on the curve: ecnXXXset gives O)."""
    rng = random.Random(2561 if curve == "NIST256" else 2551)
    if curve == "NIST256":
        p, G, n = EO.P, EO.G, EO.N
        xm, ym = _p256_xmin()
        on = {"G": G, "-G": EO.neg(G), "kG": EO.mul(rng.randrange(2, n - 1)), "(0,sqrt b)": (0, SQRT_B),
              "(0,-sqrt b)": (0, p - SQRT_B), "(xmin,y)": (xm, ym), "(xmin,-y)": (xm, p - ym)}
        noncanon = {"(p,sqrt b)": (p, SQRT_B), "(p,-sqrt b)": (p, p - SQRT_B), "(xmin+p,y)": (xm + p, ym)}
        off = {"(0,0)": (0, 0), "(Gx,Gy+1)": (G[0], G[1] + 1), "(2^256-1,2^256-1)": (M256 - 1, M256 - 1)}
        return on, noncanon, off
    p, B = DO.P, DO.B
    T = _ed_torsion()
    on = {"B": B, "-B": DO.neg(B), "kB": DO.mul(rng.randrange(2, DO.L - 1))}
    on.update(T)
    on.update(("B+" + k, DO.add(B, v)) for k, v in T.items() if k != "O")
    noncanon = {}
    for k in ["B", "-B", "kB"] + list(T):
        x, y = on[k]
        noncanon["%s x+p" % k] = (x + p, y)
        noncanon["%s y+p" % k] = (x, y + p)
        if y + 2 * p < M256:
            noncanon["%s y+2p" % k] = (x, y + 2 * p)
    off = {"(0,0)": (0, 0)}
    return on, noncanon, off


def _reduced(curve, P):
    p = EO.P if curve == "NIST256" else DO.P
    return (P[0] % p, P[1] % p)


def multiple(curve, k, P):
    """k P on the oracle of the signature code (small k, P on the curve); O as ecnXXXget reports it, (0, 1)."""
    P = _reduced(curve, P)
    if curve == "NIST256":
        R = EO.mul(abs(k), P)
        R = (0, 1) if R is None else R
        return EO.neg(R) if k < 0 and R != (0, 1) else R
    R = DO.mul(abs(k), P)
    return DO.neg(R) if k < 0 else R


# ---- scalars --------------------------------------------------------------------------------------------------------------
def scalars(curve, full):
    """{value: name}.  full: the whole list (2^k, 2^k - 1 for every k when full == 'all'); otherwise a short one."""
    n = EO.N if curve == "NIST256" else DO.L
    rng = random.Random(7 if curve == "NIST256" else 8)
    s = {}

    def put(v, name):
        if 0 <= v < M256:
            s.setdefault(v, name)
    short = [0, 1, 2, 3, 7, 8, 9, 16, 17]
    for v in (range(18) if full else short):
        put(v, str(v))
    for d in ((-2, -1, 0, 1, 2) if full else (-1, 0, 1)):
        put(n + d, "n%+d" % d if d else "n")
    for m in ((2, 4, 8) if full else (8,)):
        put(m * n, "%dn" % m)
    put(M256 - 1, "2^256-1")
    put(M256 - n, "2^256-n")
    for pat in (("88", "77", "78", "87", "f0", "0f") if full else ("88", "77")):
        put(nib(pat), "0x%s.." % pat)
    if full:
        put((n - 1) // 2, "(n-1)/2")
        put((n + 1) // 2, "(n+1)/2")
        put(1 << 255, "0x80..0")
        put((1 << 255) - 1, "0x7f..f")
    for par in (0, 1):
        for i in range(3 if full else 1):
            put(rng.randrange(M256) & ~1 | par, "random %s %d" % ("odd" if par else "even", i))
    if full:
        for k in (range(256) if full == "all" else range(7, 256, 31)):
            put(1 << k, "2^%d" % k)
            put((1 << k) - 1, "2^%d-1" % k)
    return s


# ---- the row sets ---------------------------------------------------------------------------------------------------------
def ecnmul_rows(curve):
    """[(label, e, x, y)]"""
    on, noncanon, off = points(curve)
    gen = "G" if curve == "NIST256" else "B"
    rows, seen = [], set()
    for kind, pts in (("on", on), ("noncanon", noncanon), ("off", off)):
        for name, (x, y) in pts.items():
            full = "all" if name == gen else (True if kind == "on" and not name.startswith("B+") else False)
            for e, ename in scalars(curve, full).items():
                if (e, x, y) not in seen:
                    seen.add((e, x, y))
                    rows.append(("P=%s e=%s" % (name, ename), e, x, y))
    return rows


RELATIONS = [("O", None), ("P", 1), ("-P", -1), ("2P", 2), ("-2P", -2), ("3P", 3), ("-3P", -3)]


def _ef_pairs(n, rng, full, shared_tops):
    r = lambda: rng.randrange(1, n)
    e1, e2 = r(), r()
    out = [("1,1", 1, 1), ("1,n-1", 1, n - 1), ("e,e", e1, e1), ("e,n-e", e2, n - e2), ("n,n", n, n)]
    if full:
        out += [("2^256-1,2^256-1", M256 - 1, M256 - 1), ("0,f", 0, r()), ("e,0", r(), 0),
                ("0x55..,0xaa..", nib("55"), nib("aa"))]
    if shared_tops:
        for j in (1, 8, 64, 127):                # top 2j bits equal: with Q = -P the first j digits add O
            e = rng.randrange(M256)
            low = 256 - 2 * j
            out.append(("top %d digits shared" % j, e, (e >> low << low) | rng.randrange(1 << low)))
    return out


def ecnmul2_rows(curve):
    """[(label, e, x1, y1, f, x2, y2, relation)]; relation: the k of Q = kP, None for Q = O given off the curve, or
    the name of a torsion point."""
    on, noncanon, off = points(curve)
    n = EO.N if curve == "NIST256" else DO.L
    rng = random.Random(22 if curve == "NIST256" else 23)
    O_in = (0, 0)                                # not on either curve: ecnXXXset gives O
    rows, seen = [], set()

    def add(pname, P, qname, Q, rel, full, tops):
        if (P, Q) in seen:
            return
        seen.add((P, Q))
        for lab, e, f in _ef_pairs(n, rng, full, tops):
            rows.append(("P=%s Q=%s (e,f)=(%s)" % (pname, qname, lab), e, P[0], P[1], f, Q[0], Q[1], rel))
    for kind, pts in (("on", on), ("noncanon", noncanon), ("off", off)):
        for pname, P in pts.items():
            if kind == "noncanon" and not (curve == "NIST256" or pname.startswith(("B ", "O "))):
                continue
            full = not pname.startswith("B+")
            for qname, k in RELATIONS:
                if k is None:
                    add(pname, P, qname, O_in, None, full, False)
                elif kind != "off":
                    add(pname, P, qname, multiple(curve, k, P), k, full, k == -1)
    if curve == "ED25519":
        T = _ed_torsion()
        for pname in ("B", "kB", "B+1T8", "1T8"):
            for tname, Tq in T.items():
                add(pname, on[pname], tname, Tq, tname, False, False)
    return rows


def ecdsa_rows():
    """[(label, h, r, s, qx, qy, kind)]; kind: 'valid' (valid by construction), 'R=O' (u1 G + u2 Q = O), 'h+n',
    's+1', 'h+1' (the valid row changed), 'x=p' (a key with x = p: reject)."""
    n, p = EO.N, EO.P
    rng = random.Random(256)
    keys = [("%sG" % nm, t, EO.mul(t)) for nm, t in (("1", 1), ("2", 2), ("3", 3), ("4", 4), ("5", 5), ("(n-1)", n - 1),
                                                     ("(n-2)", n - 2), ("(n-3)", n - 3), ("((n+1)/2)", (n + 1) // 2))]
    keys += [("(0,sqrt b)", None, (0, SQRT_B)), ("(0,-sqrt b)", None, (0, p - SQRT_B))]
    us = [1, 2, 3, rng.randrange(n), rng.randrange(n)]
    rows = []
    for kname, t, Q in keys:
        combos = []
        for i, u in enumerate(us):
            un = "u%d" % i
            if t is not None:
                combos += [("t %s,%s" % (un, un), t * u % n, u), ("-t %s,%s" % (un, un), -t * u % n, u)]
            combos += [("0,%s" % un, 0, u), ("%s,1" % un, u, 1)]
        combos += [("1,1", 1, 1), ("2,2", 2, 2)]
        seen = set()
        for cname, u1, u2 in combos:
            if (u1, u2) in seen:
                continue
            seen.add((u1, u2))
            lab = "Q=%s (u1,u2)=(%s)" % (kname, cname)
            R = EO.mul2(u1, EO.G, u2, Q)
            w = pow(u2, -1, n)
            if R is None:
                r = rng.randrange(1, n)
                s = r * w % n
                rows.append((lab, u1 * s % n, r, s, Q[0], Q[1], "R=O"))
                continue
            r = R[0] % n
            if r == 0:                                             # R = (0, +-sqrt b): no signature has r = 0
                continue
            s = r * w % n
            h = u1 * s % n
            rows.append((lab, h, r, s, Q[0], Q[1], "valid"))
            if h + n < M256:
                rows.append((lab + " h+n", h + n, r, s, Q[0], Q[1], "h+n"))
            rows.append((lab + " s+1", h, r, s + 1, Q[0], Q[1], "s+1"))
            rows.append((lab + " h+1", h + 1, r, s, Q[0], Q[1], "h+1"))
            if t is None and cname in ("u0,1", "u3,1"):           # the same signature under the key given as x = p
                rows.append((lab + " key x=p", h, r, s, p, Q[1], "x=p"))
    return rows


def _le(v, nb):
    return v.to_bytes(nb, "little")


def eddsa_rows():
    """[(label, h 64 bytes, sig 64 bytes, pk 32 bytes, kind)]; kind: 'eq' (R = enc([S]B - [k]A)), 'flip' (that R with
    its sign bit flipped), 'noncanon' (a key with y >= p or x = 0 with the sign bit: reject)."""
    L = DO.L
    B = DO.B
    rng = random.Random(25519)
    T = _ed_torsion()
    keys = {"B": B, "-B": DO.neg(B), "2B": DO.mul(2), "3B": DO.mul(3)}
    keys.update(T)
    keys.update(("B+" + k, DO.add(B, v)) for k, v in T.items() if k != "O")
    hs = []
    for k in (0, 1, 2, 3, L - 2, L - 1):
        hs += [("k=%s" % k if k < 4 else "k=L%+d" % (k - L), k), ("h=k+L k=%s" % (k if k < 4 else "L%+d" % (k - L)), k + L)]
    hs.append(("h=2^512-1", (1 << 512) - 1))
    Ss = [("0", 0), ("1", 1), ("2", 2), ("L-1", L - 1), ("rand0", rng.randrange(L)), ("rand1", rng.randrange(L))]
    rows = []
    i = 0
    for aname, A in keys.items():
        enc_a = DO.encode(A)
        for hname, h in hs:
            for sname, S in (Ss[i % 6], Ss[(i + 3) % 6]):
                Rp = DO.mul2(S, B, h % L, DO.neg(A))
                R = DO.encode(Rp)
                lab = "A=%s %s S=%s" % (aname, hname, sname)
                if Rp == DO.IDENTITY:
                    lab += " R'=O"
                rows.append((lab, _le(h, 64), R + _le(S, 32), enc_a, "eq"))
                flip = bytearray(R)
                flip[31] ^= 0x80
                rows.append((lab + " R sign flipped", _le(h, 64), bytes(flip) + _le(S, 32), enc_a, "flip"))
                i += 1
    # keys that decode only leniently: y = p + 1 (O), y = p ((+-sqrt(-1), 0) with either sign), y = p - 1 with the
    # sign bit (x = 0): each with the R that the canonical key would make valid
    p = DO.P
    for aname, A, enc_a in (("O as y=p+1", T["O"], _le(p + 1, 32)),
                            ("T4 as y=p", T["T4"], _le(p | (T["T4"][0] & 1) << 255, 32)),
                            ("-T4 as y=p", T["-T4"], _le(p | (T["-T4"][0] & 1) << 255, 32)),
                            ("T2 with the sign bit", T["T2"], _le((p - 1) | 1 << 255, 32))):
        for hname, h in hs[:4]:
            S = rng.randrange(L)
            R = DO.encode(DO.mul2(S, B, h % L, DO.neg(A)))
            rows.append(("A=%s %s S=rand" % (aname, hname), _le(h, 64), R + _le(S, 32), enc_a, "noncanon"))
    return rows


# ---- expected values: the oracles, once per module, in a process pool --------------------------------------------------
@pytest.fixture(scope="module")
def edge():
    """{group: (rows, expected)}: expected is (xo, yo) as 32-byte big-endian strings for ecnmul / ecnmul2, a bool for the
    signature groups."""
    out = {}
    jobs = []
    for curve in CURVES:
        one = field_oracle.ecnmul if curve == "NIST256" else field_oracle.ecnmul_edwards
        r1 = ecnmul_rows(curve)
        jobs.append(("ecnmul " + curve, r1, one, [(PRIME[curve], be(e), be(x), be(y)) for _, e, x, y in r1]))
        r2 = ecnmul2_rows(curve)
        jobs.append(("ecnmul2 " + curve, r2, field_oracle.ecnmul2,
                     [(PRIME[curve], be(e), be(x1), be(y1), be(f), be(x2), be(y2)) for _, e, x1, y1, f, x2, y2, _ in r2]))
    rs = ecdsa_rows()
    jobs.append(("ecdsa", rs, EO.verify, [(h, r, s, (qx, qy)) for _, h, r, s, qx, qy, _ in rs]))
    rd = eddsa_rows()
    jobs.append(("eddsa", rd, DO.verify_digest, [(h, sig, pk) for _, h, sig, pk, _ in rd]))
    with mp.get_context("spawn").Pool(min(16, os.cpu_count() or 1)) as pool:
        pending = [(g, rows, pool.starmap_async(fn, args, chunksize=8)) for g, rows, fn, args in jobs]
        for g, rows, res in pending:
            out[g] = (rows, res.get())
    return out


# ---- the host simulation --------------------------------------------------------------------------------------------------
def _build_sim(tmp_path_factory, src):
    from modarith_b200.gen.cli import generate_all
    d = tmp_path_factory.mktemp(os.path.splitext(src)[0])
    generate_all(verbose=False, outdir=str(d))           # fresh headers in a scratch directory, not in the source tree
    out = str(d / ("lib%s.so" % os.path.splitext(src)[0]))
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-w", "-I", str(d),
                           "-I", os.path.join(ROOT, "modarith_b200", "csrc"),
                           "-o", out, os.path.join(ROOT, "tests", "hostsim", src)])
    return ctypes.CDLL(out)


@pytest.fixture(scope="module")
def sim_ecdsa(tmp_path_factory):
    """g++ build of tests/hostsim/hostsim_ecdsa.cpp: Ecdsa::verify with the PTX blocks transcribed to C."""
    lib = _build_sim(tmp_path_factory, "hostsim_ecdsa.cpp")
    lib.sim_NIST256_ecdsa_verify.restype = ctypes.c_int
    return lib


@pytest.fixture(scope="module")
def sim_eddsa(tmp_path_factory):
    """g++ build of tests/hostsim/hostsim_eddsa.cpp: Eddsa::verify with the PTX blocks transcribed to C."""
    lib = _build_sim(tmp_path_factory, "hostsim_eddsa.cpp")
    lib.sim_ED25519_eddsa_verify.restype = ctypes.c_int
    return lib


def _args(group, row):
    """The byte-string arguments of one row, in the order of the entry point."""
    if group.startswith("ecnmul2"):
        return [be(v) for v in row[1:7]]
    if group.startswith("ecnmul"):
        return [be(v) for v in row[1:4]]
    if group == "ecdsa":
        return [be(v) for v in row[1:6]]
    return list(row[1:4])


def _check(rows, got, want):
    """Every row as the oracle says; otherwise the number of wrong rows and the labels of the first 20."""
    assert len(got) == len(rows)
    bad = [rows[i][0] for i in range(len(rows)) if got[i] != want[i]]
    assert not bad, "%d of %d rows differ from the oracle: %s" % (len(bad), len(rows), bad[:20])


# ---- the sets contain what they claim ------------------------------------------------------------------------------------
def test_edge_sets_contain_what_they_claim(edge):
    p, n = EO.P, EO.N
    # P-256: the x = 0 points and the smallest positive x are on the curve, nothing lies in between
    for x, y in ((0, SQRT_B), (0, p - SQRT_B)) + (_p256_xmin(),):
        assert EO.on_curve((x, y))
    xm = _p256_xmin()[0]
    assert all(pow((x ** 3 - 3 * x + EO.B) % p, (p - 1) // 2, p) != 1 for x in range(1, xm))
    _, noncanon, off = points("NIST256")
    assert all(EO.on_curve((x % p, y % p)) and x >= p for x, y in noncanon.values())
    assert not any((y * y - x ** 3 + 3 * x - EO.B) % p == 0 for x, y in off.values())
    # Ed25519: the torsion points have orders 1, 2, 4, 4, 8, 8, 8, 8; B + T has order 8 L exactly when T has order 8
    T = _ed_torsion()
    assert len(set(T.values())) == 8 and all(DO.on_curve(t) for t in T.values())
    orders = {k: _order(lambda a, b: DO.add(a, b), DO.IDENTITY, t) for k, t in T.items()}
    assert sorted(orders.values()) == [1, 2, 4, 4, 8, 8, 8, 8]
    for k, t in T.items():
        assert DO.mul(DO.L, DO.add(DO.B, t)) == DO.mul(DO.L % orders[k], t)
    _, nc_ed, _ = points("ED25519")
    assert all(DO.on_curve(_reduced("ED25519", P)) and max(P) >= DO.P for P in nc_ed.values())
    assert nc_ed["O y+2p"] == (0, 1 + 2 * DO.P) and len(nc_ed) == 2 * 11 + 3
    # every Q relation of the ecnmul2 rows, on the other oracle (field_oracle.ecnmul with a small scalar)
    for curve in CURVES:
        rows, _ = edge["ecnmul2 " + curve]
        nq = EO.N if curve == "NIST256" else 8 * DO.L           # the order of the whole group: -1 is nq - 1 everywhere
        one = field_oracle.ecnmul if curve == "NIST256" else field_oracle.ecnmul_edwards
        rels, checked = set(), set()
        for lab, e, x1, y1, f, x2, y2, rel in rows:
            if (x1, y1, x2, y2, rel) in checked:                # one check per distinct (P, Q, relation)
                continue
            checked.add((x1, y1, x2, y2, rel))
            if isinstance(rel, int):
                want = one(PRIME[curve], be(rel % nq), be(x1), be(y1))
                assert (be(x2), be(y2)) == want, lab
            elif rel is None:
                assert one(PRIME[curve], be(1), be(x2), be(y2)) == (be(0), be(1)), lab
            else:
                assert (x2, y2) == T[rel], lab
            rels.add(rel)
        assert {k for _, k in RELATIONS} <= rels
        if curve == "ED25519":
            assert set(T) <= rels
        assert any("top 127 digits shared" in r[0] for r in rows) and any("(e,f)=(n,n)" in r[0] for r in rows)
    # the scalars: every 2^k and 2^k - 1 on the generators, the multiples of n below 2^256
    for curve, gen in (("NIST256", EO.G), ("ED25519", DO.B)):
        es = {e for _, e, x, y in edge["ecnmul " + curve][0] if (x, y) == gen}
        assert all((1 << k) in es and (1 << k) - 1 in es for k in range(256))
        nq = EO.N if curve == "NIST256" else DO.L
        assert {nq - 2, nq - 1, nq, nq + 1, nq + 2, M256 - 1, M256 - nq, nib("88"), nib("77")} <= es
        assert (8 * nq in es) == (curve == "ED25519")
        assert {e & 1 for e in es} == {0, 1}
    # ECDSA: valid rows by construction, R = O rows, and the oracle agrees with the construction
    rows, want = edge["ecdsa"]
    kinds = [r[-1] for r in rows]
    for kind, ok in (("valid", True), ("h+n", True), ("R=O", False), ("s+1", False), ("h+1", False), ("x=p", False)):
        got = [w for k, w in zip(kinds, want) if k == kind]
        assert got and all(w == ok for w in got), kind
    assert sum(r[4] == 0 for r in rows) > 0                     # the x = 0 keys
    # Ed25519: R' = O rows among the valid ones, flipped R never valid, non-canonical keys rejected
    rows, want = edge["eddsa"]
    assert all(w for r, w in zip(rows, want) if r[-1] == "eq")
    assert not any(w for r, w in zip(rows, want) if r[-1] in ("flip", "noncanon"))
    assert sum("R'=O" in r[0] for r in rows) >= 10
    assert sum(r[-1] == "noncanon" for r in rows) == 16
    assert {g: len(edge[g][0]) for g in GROUPS} == ROWS
    assert sum(ROWS.values()) < 7000


# ---- without a GPU: the host simulation -------------------------------------------------------------------------------------
def _sim_point(fn, args):
    xo, yo = ctypes.create_string_buffer(32), ctypes.create_string_buffer(32)
    fn(*args, xo, yo)
    return xo.raw[:32], yo.raw[:32]


@pytest.mark.parametrize("curve", CURVES)
def test_hostsim_ecnmul_edge_rows(hostsim, edge, curve):
    rows, want = edge["ecnmul " + curve]
    fn = getattr(hostsim, "sim_%s_ecnmul" % curve)
    got = [_sim_point(fn, _args("ecnmul", r)) for r in rows]
    _check(rows, got, want)


@pytest.mark.parametrize("curve", CURVES)
def test_hostsim_ecnmul2_edge_rows(hostsim, edge, curve):
    rows, want = edge["ecnmul2 " + curve]
    fn = getattr(hostsim, "sim_%s_ecnmul2" % curve)
    got = [_sim_point(fn, _args("ecnmul2", r)) for r in rows]
    _check(rows, got, want)


def test_hostsim_ecdsa_edge_rows(sim_ecdsa, edge):
    rows, want = edge["ecdsa"]
    got = [bool(sim_ecdsa.sim_NIST256_ecdsa_verify(*_args("ecdsa", r))) for r in rows]
    _check(rows, got, want)


def test_hostsim_eddsa_edge_rows(sim_eddsa, edge):
    rows, want = edge["eddsa"]
    got = [bool(sim_eddsa.sim_ED25519_eddsa_verify(*_args("eddsa", r))) for r in rows]
    _check(rows, got, want)


# ---- on the GPU ------------------------------------------------------------------------------------------------------------
def _columns(group, rows):
    """The rows as the entry point's [n, w] uint8 arrays."""
    cols = list(zip(*(_args(group, r) for r in rows)))
    return [np.frombuffer(b"".join(c), dtype=np.uint8).reshape(len(rows), -1).copy() for c in cols]


def _run(group, arrays, offset=0):
    """The group's entry point on device copies of the arrays (at `offset` bytes past a 16-byte boundary); the results
    as numpy arrays: (xo, yo) for the scalar multiplications, ok for the verifiers."""
    import torch
    from modarith_b200 import ecdsa, ecn, eddsa

    def dev(a):
        buf = torch.zeros(a.size + offset, dtype=torch.uint8, device="cuda")
        v = buf[offset:].view(a.shape)
        v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        assert v.data_ptr() % 16 == offset
        return v
    d = [dev(a) for a in arrays]
    if group.startswith("ecnmul"):
        xo, yo = dev(np.zeros_like(arrays[0])), dev(np.zeros_like(arrays[0]))
        fn = ecn.ecnmul2 if group.startswith("ecnmul2") else ecn.ecnmul
        fn(group.split()[1], *d, xo=xo, yo=yo)
        torch.cuda.synchronize()
        return xo.cpu().numpy(), yo.cpu().numpy()
    ok = (ecdsa if group == "ecdsa" else eddsa).verify_digest(*d)
    torch.cuda.synchronize()
    return ok.cpu().numpy()


def _as_rows(group, res):
    if group.startswith("ecnmul"):
        xo, yo = res
        return [(xo[i].tobytes(), yo[i].tobytes()) for i in range(xo.shape[0])]
    return [bool(v) for v in res]


@pytest.mark.gpu
@pytest.mark.parametrize("group", GROUPS)
def test_gpu_edge_rows(edge, group):
    rows, want = edge[group]
    _check(rows, _as_rows(group, _run(group, _columns(group, rows))), want)


@pytest.mark.gpu
@pytest.mark.parametrize("group", GROUPS)
def test_gpu_edge_rows_tiled(edge, group):
    """The set tiled to 2^18 rows in a seeded permutation: every row as in the one-batch run, which the test above pins
    to the oracle."""
    rows, _ = edge[group]
    cols = _columns(group, rows)
    small = _run(group, cols)
    idx = np.random.Generator(np.random.PCG64(GROUPS.index(group))).permutation(NTILE) % len(rows)
    big = _run(group, [c[idx] for c in cols])
    if group.startswith("ecnmul"):
        bad = np.nonzero(~(np.all(big[0] == small[0][idx], axis=1) & np.all(big[1] == small[1][idx], axis=1)))[0]
    else:
        bad = np.nonzero(big != small[idx])[0]
    assert [(int(k), rows[idx[k]][0]) for k in bad[:10]] == []


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [1, 4, 8])
@pytest.mark.parametrize("group", GROUPS[:4])
def test_gpu_edge_rows_misaligned(edge, group, offset):
    """Inputs and outputs at a byte offset from a 16-byte boundary: the byte, word and uint2 load / store paths."""
    rows, want = edge[group]
    _check(rows, _as_rows(group, _run(group, _columns(group, rows), offset)), want)
