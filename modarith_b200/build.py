"""Generate the field headers and compile libmodarith_b200.so for sm_100a, in-tree.

The reference's build step is "run the generator, compile what it printed"
(pseudo.py:1694-1702, 1895-1903); ours is the same with nvcc:

    python -m modarith_b200.build            # regenerate + compile if stale
    python -m modarith_b200.build --force
    python -m modarith_b200.build --prime NIST384            # add-on library for another modulus of the reference's
    python -m modarith_b200.build --prime MYP="2**414-17"    # tables, or for any prime given as an expression
    python -m modarith_b200.build --prime M383="2**383-187" --a24 516287 --cof 3 --generator 12   # with its ladder
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libmodarith_b200.so")
OBJDIR = os.path.join(PKG, "build")

NVCC_FLAGS = ["-I", CSRC, "-I", os.path.join(PKG, "..", "include"), "-I", OBJDIR, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]
UNITS = ["mab_capi_X25519.cu", "mab_capi_X448.cu", "mab_capi_NIST256.cu", "mab_capi_SECP256K1.cu",
         "mab_capi_NIST256ORDER.cu", "mab_runtime.cu", "mab_jit.cu"]
# headers handed to NVRTC by mab_<P>_modprog_jit: embedded in the library as text (csrc/mab_jit.h)
JIT_COMMON = ["mab_common.cuh", "mab_field.cuh"]
JIT_FIELDS = ["X25519", "X448", "NIST256", "SECP256K1", "NIST256ORDER"]


def _as_literal(sym, text):
    """A C++ array initialised from adjacent raw string literals (chunks of whole lines, each far below any
    compiler's literal limit)."""
    assert ')MABJIT"' not in text
    out, chunk, size = ["static const char %s[] =" % sym], [], 0
    for line in text.splitlines(keepends=True):
        chunk.append(line)
        size += len(line)
        if size > 8000:
            out.append('R"MABJIT(' + "".join(chunk) + ')MABJIT"')
            chunk, size = [], 0
    out.append('R"MABJIT(' + "".join(chunk) + ')MABJIT";')
    return "\n".join(out) + "\n"


def _write_if_changed(path, text):
    if not os.path.exists(path) or open(path).read() != text:
        with open(path, "w") as f:
            f.write(text)


def write_jit_sources():
    os.makedirs(OBJDIR, exist_ok=True)
    text = "".join(_as_literal("kJitSrc_" + fn.split(".")[0], open(os.path.join(CSRC, fn)).read()) for fn in JIT_COMMON)
    _write_if_changed(os.path.join(OBJDIR, "jit_src_common.inc"), text)
    for P in JIT_FIELDS:
        src = open(os.path.join(CSRC, "gen", "field_%s.cuh" % P)).read()
        _write_if_changed(os.path.join(OBJDIR, "jit_src_%s.inc" % P), _as_literal("kJitSrc_field", src))


def _nvcc():
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built")


def _digest():
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    roots = [CSRC, os.path.join(CSRC, "gen"), os.path.join(OBJDIR, "gen"), os.path.join(PKG, "..", "include")]
    for root in filter(os.path.isdir, roots):
        for fn in sorted(os.listdir(root)):
            p = os.path.join(root, fn)
            if os.path.isfile(p) and fn.endswith((".cu", ".cuh", ".inc", ".h")):
                h.update(fn.encode())
                h.update(open(p, "rb").read())
    return h.hexdigest()


def build(force=False, verbose=True):
    from .gen.cli import generate_all
    generate_all(verbose=False)
    stamp = os.path.join(OBJDIR, "digest.txt")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    os.makedirs(OBJDIR, exist_ok=True)
    write_jit_sources()
    nvcc = _nvcc()

    def compile_one(unit):
        obj = os.path.join(OBJDIR, unit.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-Xptxas", "-v", "-c", os.path.join(CSRC, unit), "-o", obj]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        with open(obj + ".log", "w") as f:
            f.write(r.stdout)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (unit, r.stdout[-4000:]))
        return obj

    with cf.ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(compile_one, UNITS))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
    subprocess.check_call(cmd)
    with open(stamp, "w") as f:
        f.write(dig)
    if verbose:
        print("built", LIB)
    return LIB


def extra_lib_path(name):
    return os.path.join(PKG, "libmodarith_b200_%s.so" % name)


def build_extra(name, expr=None, force=False, verbose=True, curve=None):
    """An add-on library with the field entry points (mab_<NAME>_modmul, ..., _modprog, _modprog_jit) for a modulus
    that is not one of the five built in: the reference's `python3 monty.py 64 NIST384` + compile, in one step
    (pseudo.py:1694-1702).  Same C ABI, same kernels (csrc/mab_capi.inc instantiated on the generated header), linked
    with the library's own runtime objects so that it stands alone: modarith_b200/libmodarith_b200_<NAME>.so, which
    Field(NAME) loads.  `expr`: a Python integer expression for a modulus the tables do not name.
    `curve` = (a24, cof, generator): the modulus carries a Montgomery curve B y^2 = x^3 + A x^2 + x with
    a24 = (A - 2) / 4 and cofactor 2^cof -- the constants a user adds to rfc7748.c:117-132 for a curve of their own --
    and the library also exports the ladder entry points mab_<NAME>_rfc7748[_perkey|_validate|_host|_host_multi]."""
    import re
    from .gen.cli import generate
    from .primes import Prime, named
    if not re.fullmatch(r"[A-Za-z][A-Za-z0-9]*", name):
        raise ValueError("a modulus name is an identifier (it becomes part of the C symbols): %r" % name)
    if expr is not None:
        p = eval(expr, {"__builtins__": {}})
        P = Prime(name, int(p), "monty")
    else:
        P = named(name)
    if curve is not None:
        a24, cof, gen = (int(v) for v in curve)
        if not (0 < a24 < 2**31 and cof in (2, 3) and 0 < gen < 2**31):
            raise ValueError("curve constants: 0 < a24 < 2^31, cof 2 or 3 (rfc7748.c:121-131), 0 < generator < 2^31")
        if P.nbytes % 4 != 0:
            raise ValueError("the ladder kernels move whole 32-bit words: a curve needs a modulus of 32k-24 .. 32k bits "
                             "(Nbytes = %d here)" % P.nbytes)
        P = Prime(P.name, P.p, P.family, a24=a24, cof=cof, generator=gen)
    build(verbose=False)                                   # the runtime objects and the common JIT sources
    ext = os.path.join(OBJDIR, "ext")
    os.makedirs(ext, exist_ok=True)
    hdr = os.path.join(ext, "field_%s.cuh" % name)
    generate(P, hdr, verbose=False)
    unit = os.path.join(ext, "mab_capi_%s.cu" % name)
    _write_if_changed(unit, '// C ABI instantiation for %s (python -m modarith_b200.build --prime)\n#include "field_%s.cuh"\n'
                      '#include "modarith_b200.h"\nextern "C" {\nMAB_DECLARE_FIELD(%s)      // exported like the built-in moduli\n%s}\n'
                      '#define MAB_P %s\n#define MAB_F F_%s\n%s#define MAB_JIT_SRC "jit_src_%s.inc"\n#include "mab_capi.inc"\n'
                      % (name, name, name, "MAB_DECLARE_CURVE(%s)\n" % name if curve else "", name, name,
                         "#define MAB_HAS_CURVE 1\n" if curve else "", name))
    _write_if_changed(os.path.join(ext, "jit_src_%s.inc" % name), _as_literal("kJitSrc_field", open(hdr).read()))
    out = extra_lib_path(name)
    stamp = os.path.join(ext, "digest_%s.txt" % name)
    dig = hashlib.sha256((_digest() + open(hdr).read() + open(unit).read()).encode()).hexdigest()
    if not force and os.path.exists(out) and os.path.exists(stamp) and open(stamp).read() == dig:
        return out
    nvcc = _nvcc()
    obj = os.path.join(ext, "mab_capi_%s.o" % name)
    cmd = [nvcc] + NVCC_FLAGS + ["-I", ext, "-Xptxas", "-v", "-c", unit, "-o", obj]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    with open(obj + ".log", "w") as f:
        f.write(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (unit, r.stdout[-4000:]))
    subprocess.check_call([nvcc, "-shared", "-o", out, obj, os.path.join(OBJDIR, "mab_runtime.o"), os.path.join(OBJDIR, "mab_jit.o"),
                           "-gencode", "arch=compute_100a,code=sm_100a", "-ldl"])
    with open(stamp, "w") as f:
        f.write(dig)
    if verbose:
        print("built", out)
    return out


if __name__ == "__main__":
    if "--prime" in sys.argv:
        spec = sys.argv[sys.argv.index("--prime") + 1]
        nm, _, ex = spec.partition("=")

        def opt(flag, default=None):
            return sys.argv[sys.argv.index(flag) + 1] if flag in sys.argv else default
        cv = None
        if "--a24" in sys.argv:
            cv = (int(opt("--a24")), int(opt("--cof", "3")), int(opt("--generator", "9")))
        build_extra(nm, ex or None, force="--force" in sys.argv, curve=cv)
    else:
        build(force="--force" in sys.argv)
