"""ctypes binding of libmodarith_b200.so (include/modarith_b200.h).

The reference binds its generated functions the same way (ctypes.CDLL on test.so,
pseudo.py:1704-1750).  There is NO CPU fallback: if the CUDA library has not been built
(python -m modarith_b200.build) or cannot be loaded, importing a field raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_int, c_size_t, c_uint, c_void_p, POINTER, c_float, c_double, c_longlong

PKG = os.path.dirname(os.path.abspath(__file__))
# MODARITH_B200_LIB selects an alternative build of the SAME library (kernel-tuning experiments,
# tools/variants.py); it is never a different backend.
LIBPATH = os.environ.get("MODARITH_B200_LIB") or os.path.join(PKG, "libmodarith_b200.so")

PRIMES = ("X25519", "X448", "NIST256", "SECP256K1", "NIST256ORDER")
CURVES = ("X25519", "X448")

_P = c_void_p          # device pointers travel as integers
_TAIL = [c_size_t, c_size_t, c_void_p]      # n, stride, stream

# name -> leading argument types (the reference's argument order), SURVEY.md 8a
FIELD_SIGNATURES = {
    "info": [POINTER(c_int)] * 8,
    "modfsb": [_P, _P],
    "modadd": [_P, _P, _P],
    "modsub": [_P, _P, _P],
    "modneg": [_P, _P],
    "modmul": [_P, _P, _P],
    "modsqr": [_P, _P],
    "bench_modmul": [_P, _P, _P, c_uint],
    "modmli": [_P, c_int, _P],
    "modcpy": [_P, _P],
    "modnsqr": [_P, c_int],
    "modpro": [_P, _P],
    "modinv": [_P, _P, _P],
    "modinv_perelement": [_P, _P],
    "modqr": [_P, _P, _P],
    "modsqrt": [_P, _P, _P],
    "modis1": [_P, _P],
    "modis0": [_P, _P],
    "modzer": [_P],
    "modone": [_P],
    "modint": [c_int, _P],
    "nres": [_P, _P],
    "redc": [_P, _P],
    "modcsw": [_P, _P, _P],
    "modcmv": [_P, _P, _P],
    "modshl": [c_uint, _P],
    "modshr": [c_uint, _P, _P],
    "modhaf": [_P],
    "mod2r": [c_uint, _P],
    "modexp": [_P, _P],
    "modimp": [_P, _P, _P],
    "modsign": [_P, _P],
    "modcmp": [_P, _P, _P],
}


class mab_insn(ctypes.Structure):
    """include/modarith_b200.h: one instruction of a mab_<P>_modprog program."""
    _fields_ = [("op", ctypes.c_ubyte), ("dst", ctypes.c_ubyte), ("a", ctypes.c_ubyte), ("b", ctypes.c_ubyte),
                ("imm", ctypes.c_uint32)]


OPCODES = {n: i for i, n in enumerate(("add", "sub", "neg", "mul", "sqr", "mli", "cpy", "nsqr", "pro", "inv", "sqrt",
                                       "zer", "one", "int", "haf"))}
PROG_NREG, PROG_MAX = 16, 320
ERR_NOJIT, ERR_JIT = 100003, 100004

_lib = None


class MabError(RuntimeError):
    pass


def _bind_field(lib, P):
    """argtypes / restype of every mab_<P>_* field entry point (include/modarith_b200.h, MAB_DECLARE_FIELD)."""
    for name, lead in FIELD_SIGNATURES.items():
        fn = getattr(lib, "mab_%s_%s" % (P, name))
        fn.argtypes = lead + ([] if name == "info" else _TAIL)
        fn.restype = c_int
    for name in ("modprog", "modprog_jit"):
        fn = getattr(lib, "mab_%s_%s" % (P, name))
        fn.argtypes = [POINTER(mab_insn), c_size_t, POINTER(c_void_p), c_int, POINTER(c_void_p), POINTER(ctypes.c_ubyte),
                       c_int, c_size_t, c_size_t, c_void_p]
        fn.restype = c_int
    fn = getattr(lib, "mab_%s_modprog_cubin" % P)
    fn.argtypes = [POINTER(mab_insn), c_size_t, c_int, POINTER(ctypes.c_ubyte), c_int, c_void_p, POINTER(c_size_t)]
    fn.restype = c_int


def _bind_curve(lib, P):
    """The ladder entry points of one curve (include/modarith_b200.h, MAB_DECLARE_CURVE)."""
    for name in ("rfc7748", "rfc7748_perkey", "rfc7748_validate"):
        fn = getattr(lib, "mab_%s_%s" % (P, name))
        fn.argtypes = [_P, _P, _P, c_size_t, c_void_p]
        fn.restype = c_int
    for name in ("rfc7748_host", "rfc7748_host_multi"):
        fn = getattr(lib, "mab_%s_%s" % (P, name))
        fn.argtypes = [c_void_p, c_void_p, c_void_p, c_size_t, c_int]
        fn.restype = c_int


_extra = {}


def extra_lib_path(prime: str) -> str:
    return os.path.join(PKG, "libmodarith_b200_%s.so" % prime)


def load_for(prime: str) -> ctypes.CDLL:
    """The library that holds mab_<prime>_*: the shipped one for the built-in moduli, otherwise the add-on library
    `python -m modarith_b200.build --prime <prime>` produced.  Fails loudly when neither exists."""
    if prime in PRIMES:
        return load()
    if prime in _extra:
        return _extra[prime]
    path = extra_lib_path(prime)
    if not os.path.exists(path):
        raise MabError("no library for modulus %r: the built-in ones are %s; build an add-on library with "
                       "`python -m modarith_b200.build --prime %s` (or --prime %s=<expression>)"
                       % (prime, ", ".join(PRIMES), prime, prime))
    lib = ctypes.CDLL(path)
    lib.mab_error_string.restype = c_char_p
    lib.mab_error_string.argtypes = [c_int]
    lib.mab_jit_log.restype = c_char_p
    _bind_field(lib, prime)
    if hasattr(lib, "mab_%s_rfc7748" % prime):              # built with a Montgomery curve (--a24 / --cof)
        _bind_curve(lib, prime)
    _extra[prime] = lib
    return lib


def load() -> ctypes.CDLL:
    """Load the CUDA library, binding every symbol the header declares.  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBPATH):
        raise MabError("%s is missing: build it with `python -m modarith_b200.build` "
                       "(nvcc, sm_100a).  There is no CPU fallback." % LIBPATH)
    lib = ctypes.CDLL(LIBPATH)
    lib.mab_version.restype = c_char_p
    lib.mab_error_string.restype = c_char_p
    lib.mab_error_string.argtypes = [c_int]
    lib.mab_device_count.restype = c_int
    lib.mab_params.argtypes = [c_char_p] + [POINTER(c_int)] * 5
    lib.mab_products.argtypes = [c_char_p, c_char_p]
    lib.mab_products.restype = c_longlong
    lib.mab_imad_peak.argtypes = [c_int, c_int, c_int, c_int, POINTER(c_float), POINTER(c_double), c_void_p]
    lib.mab_pipe_probe.argtypes = [c_int, c_int, c_int, c_int, POINTER(c_float), POINTER(c_char_p), POINTER(c_int),
                                   POINTER(c_int), c_void_p]
    lib.mab_probe_unsat29_modmul.argtypes = [_P, _P, _P, c_uint, c_size_t, c_size_t, c_void_p]
    for P in PRIMES:
        _bind_field(lib, P)
    lib.mab_jit_log.restype = c_char_p
    lib.mab_NIST256_ecnmul.argtypes = [_P, _P, _P, _P, _P, c_size_t, c_void_p]
    lib.mab_NIST256_ecnmul.restype = c_int
    lib.mab_ED25519_ecnmul.argtypes = [_P, _P, _P, _P, _P, c_size_t, c_void_p]
    lib.mab_ED25519_ecnmul.restype = c_int
    for name in ("mab_NIST256_ecnmul2", "mab_ED25519_ecnmul2"):
        fn = getattr(lib, name)
        fn.argtypes = [_P] * 8 + [c_size_t, c_void_p]
        fn.restype = c_int
    for P in CURVES:
        _bind_curve(lib, P)
    lib.mab_NIST256_ecdsa_verify.argtypes = [_P] * 6 + [c_size_t, c_void_p]
    lib.mab_NIST256_ecdsa_verify.restype = c_int
    lib.mab_ED25519_eddsa_verify.argtypes = [_P] * 4 + [c_size_t, c_void_p]
    lib.mab_ED25519_eddsa_verify.restype = c_int
    _lib = lib
    return lib


def exported_symbols():
    """Every symbol include/modarith_b200.h declares (used by the CPU-side ABI test)."""
    syms = ["mab_version", "mab_error_string", "mab_device_count", "mab_params", "mab_products", "mab_imad_peak",
            "mab_pipe_probe", "mab_release_workspaces", "mab_probe_unsat29_modmul", "mab_jit_log",
            "mab_NIST256_ecnmul", "mab_ED25519_ecnmul", "mab_NIST256_ecnmul2", "mab_ED25519_ecnmul2"]
    for P in PRIMES:
        syms += ["mab_%s_%s" % (P, n) for n in FIELD_SIGNATURES] + ["mab_%s_modprog" % P, "mab_%s_modprog_jit" % P, "mab_%s_modprog_cubin" % P]
    for P in CURVES:
        syms += ["mab_%s_rfc7748" % P, "mab_%s_rfc7748_host" % P, "mab_%s_rfc7748_validate" % P,
                 "mab_%s_rfc7748_perkey" % P, "mab_%s_rfc7748_host_multi" % P]
    return syms


def signature_symbols():
    """Every symbol include/modarith_b200_sig.h declares."""
    return ["mab_NIST256_ecdsa_verify", "mab_ED25519_eddsa_verify"]


def check(code: int, what: str = "", lib=None):
    if code != 0:
        lib = lib or load()
        msg = lib.mab_error_string(code).decode()
        if code in (ERR_NOJIT, ERR_JIT):
            msg += "\n" + lib.mab_jit_log().decode(errors="replace")[-4000:]
        raise MabError("%s failed: %s (code %d)" % (what or "modarith_b200 call", msg, code))


def params(prime: str):
    lib = load_for(prime)
    v = [c_int() for _ in range(8)]
    check(getattr(lib, "mab_%s_info" % prime)(*[ctypes.byref(x) for x in v]), "mab_%s_info" % prime)
    d = dict(zip(("nlimbs", "nbits", "nbytes", "pm1d2", "pro_sqr", "pro_mul", "montgomery", "has_curve"),
                 [x.value for x in v]))
    d.update(wordlength=32, radix=32)
    return d


def products(prime: str, what: str) -> int:
    """Algorithmic 32x32->64 limb products of one call (SURVEY.md 8d)."""
    r = int(load().mab_products(prime.encode(), what.encode()))
    if r != -1 or prime in ("X25519", "X448", "NIST256"):
        return r
    q = params(prime)
    L = q["nlimbs"]
    M, S = L * L, L * (L + 1) // 2
    pro = q["pro_sqr"] * S + q["pro_mul"] * M
    k = q["pm1d2"]
    table = {"modmul": M, "modsqr": S, "modmli": L, "modpro": pro,
             "modinv": pro + (k - 1) * (S + M) + (k + 1) * S + M}
    return table.get(what, -1)
