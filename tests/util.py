"""Shared helpers for the parity tests."""
import ctypes

import numpy as np

from field_oracle import FieldOracle, rfc7748 as oracle_rfc7748  # noqa: F401
from modarith_b200.primes import ALL_PRIMES as PRIMES

SIM_OPS = ["ADD", "SUB", "NEG", "MUL", "SQR", "MLI", "NSQR", "PRO", "INV", "INVH", "QR", "QRH", "SQRT", "SQRTH",
           "IS1", "IS0", "ONE", "INT", "NRES", "REDC", "CSW", "CMV", "SHL", "SHR", "HAF", "2R", "SIGN", "CMP", "FSB",
           "IMPW", "EXPW", "MLA", "ADDTT", "SUBTT", "MULW", "SQRW", "CANON", "REDCW"]
SIM = {n: i for i, n in enumerate(SIM_OPS)}


def limbs_of(name):
    return (PRIMES[name].nbits + 31) // 32


class Sim:
    """Thin wrapper over the hostsim library: operates on Python ints through imp/exp words."""

    def __init__(self, lib, name):
        self.lib, self.name, self.L = lib, name, limbs_of(name)
        self.fn = getattr(lib, "sim_%s_op" % name)
        self.fn.restype = ctypes.c_int
        self.P = PRIMES[name]

    def _arr(self, v=None):
        A = (ctypes.c_uint32 * self.L)()
        if v is not None:
            for i in range(self.L):
                A[i] = (v >> (32 * i)) & 0xFFFFFFFF
        return A

    @staticmethod
    def _val(A):
        return sum(int(A[i]) << (32 * i) for i in range(len(A)))

    def raw(self, op, a=None, b=None, scalar=0):
        """op on STORED representations given/returned as integers."""
        r, r2 = self._arr(), self._arr()
        ret = self.fn(SIM[op], self._arr(a) if a is not None else None, self._arr(b) if b is not None else None,
                      ctypes.c_uint32(scalar), r, r2)
        return self._val(r), ret, self._val(r2)

    def imp(self, v):
        """plain integer (< 2^(32L)) -> stored form (modimp on words)."""
        r, lt, _ = self.raw("IMPW", v)
        return r, lt

    def exp(self, s):
        """stored form -> canonical plain integer (modexp on words)."""
        return self.raw("EXPW", s)[0]


def random_bytes(seed, n, nb):
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, 256, (n, nb), dtype=np.uint8)


def sample_rows(n, m, head=0):
    """Rows checked against the restatements where the reference build (oracle/_ref) is absent: the first `head`
    rows (planted corner cases) and a fixed seeded sample of m of the others, ascending."""
    rest = np.random.Generator(np.random.PCG64(n)).choice(np.arange(head, n), min(m, n - head), replace=False)
    return np.concatenate([np.arange(head), np.sort(rest)])


def ref_rfc7748_batch(lib, k, u):
    out = np.zeros_like(k)
    lib.ref_rfc7748_batch(k.ctypes.data_as(ctypes.c_char_p), u.ctypes.data_as(ctypes.c_char_p),
                          out.ctypes.data_as(ctypes.c_char_p), ctypes.c_size_t(k.shape[0]), ctypes.c_int(0))
    return out


REF_OPS = {"mul": 0, "sqr": 1, "inv": 2, "sqrt": 3, "add": 4, "sub": 5, "neg": 6, "pro": 7, "id": 8, "mli": 9,
           "haf": 10, "qr": 11}


def ref_field_batch(lib, op, a, b=None, ib=0):
    """a, b: [n, Nbytes] big-endian uint8 -> ([n, Nbytes] outputs, status[n]) via the reference's C."""
    n = a.shape[0]
    out = np.zeros_like(a)
    st = np.zeros(n, dtype=np.int32)
    lib.ref_field_batch(REF_OPS[op], a.ctypes.data_as(ctypes.c_char_p),
                        b.ctypes.data_as(ctypes.c_char_p) if b is not None else None, ctypes.c_int(ib),
                        out.ctypes.data_as(ctypes.c_char_p), st.ctypes.data_as(ctypes.POINTER(ctypes.c_int)),
                        ctypes.c_size_t(n), ctypes.c_int(0))
    return out, st


def oracle_field_op(F: FieldOracle, op, a, b=None, ib=0):
    """Value-level result of one golden-file operation; returns (value, status)."""
    p = F.p
    av, st = a % p, int(a < p)
    bv = None if b is None else b % p
    if op == "mul":
        return F.modmul(av, bv), st
    if op == "sqr":
        return F.modsqr(av), st
    if op == "inv":
        return F.modinv(av), st
    if op == "sqrt":
        return F.modsqrt(av), st
    if op == "add":
        return F.modadd(av, bv), st
    if op == "sub":
        return F.modsub(av, bv), st
    if op == "neg":
        return F.modneg(av), st
    if op == "pro":
        return F.modpro(av), st
    if op == "id":
        return av, st
    if op == "mli":
        return F.modmli(av, ib), st
    if op == "haf":
        return F.modhaf(av), st
    if op == "qr":
        return 0, F.modqr(None, av)
    raise KeyError(op)
