#!/usr/bin/env python3
"""Constant-time audit of the compiled kernels (no GPU needed): does ptxas keep what the source promises?

The reference's discipline is "no secret-dependent branch, no secret-dependent address" and its README
tells the user to inspect the compiler output (pseudo.py:984,1022; README.md:104-108).  The CUDA source
here is written that way (mask selects, masked table scans, loop counts that are public); this tool checks
the SASS that actually ships:

    python tools/ct_audit.py                       # the default kernel list, from modarith_b200/build/*.o
    python tools/ct_audit.py OBJ PATTERN [...]     # any kernel

Method: forward may-taint dataflow over the control-flow graph of each kernel.
  sources   every register written by a load from global, shared or local memory (key bytes, points, table
            entries, stashed scalars -- all of it is treated as secret), and everything computed from a
            tainted register or predicate (carry predicates included); an instruction guarded by a tainted
            predicate taints what it writes
  clean     kernel parameters and constants (LDC/LDCU/ULDC), special registers (S2R: thread and block
            indices, %smid), clocks, and the values returned by the atomics on the work counters
  flagged   (1) a branch, EXIT, or call whose guard predicate is tainted
            (2) a memory instruction with a tainted register inside its address brackets
            (3) instructions whose timing depends on operand values on this architecture (none are
                used: integer division and the like would show up here by name)
Exit status 1 if anything is flagged.  Loop counters, `idx < n` tests and the work-queue logic pass because
they are computed from clean values only; the per-element int arrays of modcsw/modcmv are loaded from memory
and therefore tainted -- they are used as masks, never as guards or indices, which is exactly what is checked.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "modarith_b200", "build")
DEFAULT = [("mab_capi_X25519.o", "k_rfc7748"), ("mab_capi_X448.o", "k_rfc7748"),
           ("mab_capi_NIST256.o", "k_ecnmul"), ("mab_capi_X25519.o", "k_ecnmul"), ("mab_capi_NIST256.o", "k_ecdsa"),
           ("mab_capi_X25519.o", "k_eddsa"),
           ("mab_capi_NIST256.o", "k_field"), ("mab_capi_X25519.o", "k_field"), ("mab_capi_X448.o", "k_field"),
           ("mab_capi_SECP256K1.o", "k_field"), ("mab_capi_NIST256ORDER.o", "k_field"),
           ("mab_capi_NIST256.o", "k_inv_shared"), ("mab_capi_X25519.o", "k_inv_shared"),
           ("mab_capi_NIST256.o", "k_prog"), ("mab_capi_X25519.o", "k_prog"), ("mab_capi_X448.o", "k_prog")]

LOADS = ("LDG", "LDS", "LDL", "LD.", "LDSM")
CLEAN_DEST = ("LDC", "LDCU", "ULDC", "S2R", "S2UR", "CS2R", "ATOM", "ATOMG", "ATOMS", "MOV32I")
NO_DEST = ("ST", "RED", "BRA", "EXIT", "BAR", "BSYNC", "BSSY", "NOP", "WARPSYNC", "MEMBAR", "ERRBAR", "YIELD", "RET",
           "CALL", "DEPBAR", "ENDCOLLECTIVE", "CCTL", "NANOSLEEP", "BREAK", "KILL", "BPT", "JMP", "BRX", "JMX")
TWO_PRED_DEST = ("ISETP", "UISETP", "PLOP3", "UPLOP3", "FSETP", "PSETP")
VARIABLE_TIME = ("IDIV", "MUFU")          # value-dependent latency would be a leak; neither appears in the field code
REG = re.compile(r"\b(UR\d+|UP\d+|R\d+|P\d+)\b")


def parse(obj, pattern):
    txt = subprocess.run(["cuobjdump", "-sass", obj], stdout=subprocess.PIPE, text=True, check=True).stdout
    for f in re.split(r"\n\s*Function : ", txt)[1:]:
        name = f.split("\n")[0].strip()
        if pattern not in name:
            continue
        ins = []
        for l in f.split("\n"):
            m = re.match(r"\s+/\*([0-9a-f]{4,6})\*/\s+(.*?)\s*;", l)
            if m:
                ins.append((int(m.group(1), 16), m.group(2)))
        yield name, ins


def width(op):
    if ".128" in op:
        return 4
    if ".64" in op or "WIDE" in op or (op.startswith("CS2R") and ".32" not in op):
        return 2
    return 1


def expand(reg, n):
    m = re.match(r"(U?R)(\d+)$", reg)
    if not m or n == 1:
        return [reg]
    return ["%s%d" % (m.group(1), int(m.group(2)) + i) for i in range(n)]


def split_operands(text):
    """'@!P0 IADD3.X R5, P0, PT, R5, R15, RZ, P0, !PT' -> (guard, opcode, [operands])"""
    guard = None
    m = re.match(r"@(!?)(U?P\d+|U?PT)\s+(.*)", text)
    if m:
        guard = m.group(1) + m.group(2)
        text = m.group(3)
    parts = text.split(None, 1)
    op = parts[0]
    ops = [o.strip() for o in parts[1].split(",")] if len(parts) > 1 else []
    return guard, op, ops


def regs_in(operand, n=1):
    out = []
    for r in REG.findall(operand):
        wide = n if (r.startswith("R") and (".64" in operand or n > 1)) else 1
        out += expand(r, max(wide, 2 if ".64" in operand and r[0] in "RU" and not r.startswith("UP") else 1)) if wide > 1 or ".64" in operand else [r]
    return out


def analyse(name, ins):
    addr_index = {a: i for i, (a, _) in enumerate(ins)}
    decoded = []
    for a, text in ins:
        guard, op, ops = split_operands(text)
        base = op.split(".")[0]
        dests, srcs = [], []
        w = width(op)
        if base.startswith(NO_DEST) and not base.startswith("STS") or base in ("STS", "STG", "STL", "ST"):
            srcs = [r for o in ops for r in regs_in(o, 1)]
            if base.startswith("ST") or base.startswith("RED"):
                srcs = []
                for k, o in enumerate(ops):
                    srcs += regs_in(o, w if (k == len(ops) - 1 and "[" not in o) else 1)
        elif base.startswith(TWO_PRED_DEST):
            dests = [r for o in ops[:2] for r in REG.findall(o)]
            srcs = [r for o in ops[2:] for r in regs_in(o)]
        elif base == "P2R":
            # P2R Rd, PR, Rs, mask: Rd = (Rs & ~mask) | (predicates & mask) -- only the predicates in the mask are read
            dests = REG.findall(ops[0])
            mask = int(ops[3], 16) if len(ops) > 3 and ops[3].startswith("0x") else 0x7f
            srcs = ["P%d" % i for i in range(7) if (mask >> i) & 1] + REG.findall(ops[2])
        elif base == "R2P":
            mask = int(ops[2], 16) if len(ops) > 2 and ops[2].startswith("0x") else 0x7f
            dests = ["P%d" % i for i in range(7) if (mask >> i) & 1]
            srcs = [r for o in ops[1:] for r in REG.findall(o)]
        else:
            k = 0
            # leading predicates (SHFL PT, R3 / ATOMG PT, R2) are destinations, then one register destination,
            # then the predicates that directly follow it (carry-outs)
            while k < len(ops) and re.fullmatch(r"U?P\d+|U?PT", ops[k]):
                dests += REG.findall(ops[k])
                k += 1
            if k < len(ops):
                d = REG.findall(ops[k])
                if d and re.fullmatch(r"U?R\d+(\.\w+)*", ops[k]):
                    dests += expand(d[0], w if base.startswith(LOADS + ("IMAD", "LDC", "MOV", "SHF", "CS2R", "UIMAD", "ULDC", "LDCU", "ATOM")) or "WIDE" in op else 1)
                    k += 1
                    while k < len(ops) and re.fullmatch(r"U?P\d+|U?PT", ops[k]):
                        dests += REG.findall(ops[k])
                        k += 1
            for j, o in enumerate(ops[k:]):
                # the 64-bit addend of a wide multiply-add is the last register operand
                n = 2 if ("WIDE" in op and j == len(ops[k:]) - 1 - (1 if re.fullmatch(r"!?U?P\w+", ops[-1]) else 0) and "[" not in o) else 1
                srcs += regs_in(o, n)
        addr_regs = []
        for o in ops:
            for br in re.findall(r"\[([^\]]*)\]", o):
                if br.startswith("UR") and "desc" in o and o.index("[" + br) == o.index("["):
                    continue                          # desc[URx] is the descriptor, not the address
                for r in REG.findall(br):
                    addr_regs += expand(r, 2 if ".64" in br else 1)
        target = None
        if base in ("BRA", "BSSY", "CALL", "JMP"):
            t = re.findall(r"0x([0-9a-f]+)", text)
            if t:
                target = addr_index.get(int(t[-1], 16))
        decoded.append(dict(addr=a, text=text, guard=guard, op=op, base=base, dests=dests, srcs=srcs, addr_regs=addr_regs,
                            target=target, branch_pred=[r for o in ops for r in REG.findall(o) if re.fullmatch(r"!?U?P\d+", o.strip())]
                            if base == "BRA" else []))
    n = len(decoded)
    # successors (CALL -> callee, RET -> the instruction after every call site: ptxas emits calls for 64-bit division)
    succ = [[] for _ in range(n)]
    returns = [i + 1 for i, d in enumerate(decoded) if d["base"] == "CALL" and i + 1 < n]
    for i, d in enumerate(decoded):
        if d["base"] == "CALL" and d["target"] is not None:
            succ[i].append(d["target"])
            continue
        if d["base"] == "RET":
            succ[i] += returns
            if d["guard"] is None:
                continue
        if d["base"] == "EXIT" and d["guard"] is None:
            continue
        if d["base"] in ("BRA", "JMP") and d["target"] is not None:
            succ[i].append(d["target"])
            if d["guard"] is None and not d["branch_pred"] and ".U" not in d["op"] and ".DIV" not in d["op"]:
                continue
        if i + 1 < n:
            succ[i].append(i + 1)
    # State = (tainted registers, conditional-clean facts).  A fact "R9?P1" says: R9 holds a clean value whenever
    # P1 is true -- what a predicated definition `@P1 IADD3.X R9, ...` with clean sources establishes when R9 held
    # secret data before.  A use guarded by the same literal (`@P1 STG [R8.64]`) may rely on it.  Facts die when the
    # register or the predicate is written again; at control-flow merges taint is united, facts are intersected.
    # ptxas parks predicates in single bits of a general register (`LOP3 R2, R2, ~bit, RZ, 0xc0` then
    # `@P LOP3 R2, R2, bit, RZ, 0xfc`, read back with `LOP3 P4, RZ, R2, bit, RZ, 0xc0`): clean loop bounds and
    # secret carries end up side by side in one register, so such registers are tracked per bit ("R2.b13").
    def anybit(t, r):
        pre = r + ".b"
        return any(x.startswith(pre) for x in t)

    def tainted(t, cc, r, guard):
        return (r in t or anybit(t, r)) and not (guard and (r + "?" + guard) in cc)

    def bit_idiom(d):
        """('and'|'or'|'test', register, mask) for the three predicate-parking forms, else None"""
        if d["base"] != "LOP3":
            return None
        _, _, ops = split_operands(d["text"])
        if len(ops) >= 6 and re.fullmatch(r"U?P\d+", ops[0]) and ops[1] == "RZ" and re.fullmatch(r"R\d+(\.reuse)?", ops[2]) \
                and ops[3].startswith("0x") and ops[4] == "RZ" and ops[5] == "0xc0":
            return ("test", ops[2].split(".")[0], int(ops[3], 16))
        if len(ops) >= 5 and re.fullmatch(r"R\d+", ops[0]) and ops[1].split(".")[0] == ops[0] and ops[2].startswith("0x") and ops[3] == "RZ":
            if ops[4] == "0xc0":
                return ("and", ops[0], int(ops[2], 16))
            if ops[4] == "0xfc":
                return ("or", ops[0], int(ops[2], 16))
        return None

    state_in = [None] * n
    state_in[0] = (frozenset(), frozenset())
    work = collections.deque([0])
    while work:
        i = work.popleft()
        d = decoded[i]
        t, cc = set(state_in[i][0]), set(state_in[i][1])
        g = d["guard"]
        gp = g.lstrip("!") if g else None
        src_t = any(tainted(t, cc, r, g) for r in d["srcs"]) or (gp in t if gp else False)
        idiom = bit_idiom(d)
        if idiom and not (idiom[1] in t):
            kind, r, mask = idiom
            if kind == "and" and g is None:
                for b in range(32):
                    if not (mask >> b) & 1:
                        t.discard("%s.b%d" % (r, b))
            elif kind == "or":
                if gp and gp in t:
                    for b in range(32):
                        if (mask >> b) & 1:
                            t.add("%s.b%d" % (r, b))
            elif kind == "test":
                hit = any(("%s.b%d" % (r, b)) in t for b in range(32) if (mask >> b) & 1) or (gp in t if gp else False)
                for pd in d["dests"]:
                    if pd.startswith(("P", "UP")):
                        if hit:
                            t.add(pd)
                        elif g is None:
                            t.discard(pd)
            if kind != "and" or g is None:
                out = (frozenset(t), frozenset(cc))
                for j in succ[i]:
                    if state_in[j] is None:
                        merged = out
                    else:
                        (ta, ca), (tb, cb) = state_in[j], out
                        keep = frozenset(f for f in (ca | cb)
                                         if (f in ca or f.split("?")[0] not in ta) and (f in cb or f.split("?")[0] not in tb))
                        merged = (ta | tb, keep)
                    if merged != state_in[j]:
                        state_in[j] = merged
                        work.append(j)
                continue
        slots = None
        if d["base"] in ("LDL", "STL"):
            # register spills: [R1 + offset] slots carry the taint of what was stored (any other local addressing
            # is treated as secret)
            m = re.search(r"\[R1(?:\+(0x[0-9a-f]+))?\]", d["text"])
            if m:
                off = int(m.group(1), 16) if m.group(1) else 0
                slots = ["L%d" % (off + 4 * k) for k in range(width(d["op"]))]
        if d["base"] == "STL" and slots:
            vals = d["srcs"][-len(slots):] if len(d["srcs"]) >= len(slots) else d["srcs"]
            vt = any(tainted(t, cc, r, g) for r in vals) or (gp in t if gp else False)
            for sl in slots:
                if vt:
                    t.add(sl)
                elif g is None:
                    t.discard(sl)
            new = False
        elif d["base"] == "LDL" and slots:
            new = any(sl in t for sl in slots) or (gp in t if gp else False)
        elif d["base"].startswith(LOADS) and ".STRONG" in d["op"] and d["base"] == "LDG":
            new = False          # volatile loads: the kernels use them for the work counters only (mab_kernels.cuh)
        elif d["base"].startswith(LOADS):
            new = True
        elif d["base"].startswith(CLEAN_DEST):
            new = (gp in t) if gp else False
        else:
            new = src_t
        for r in d["dests"]:
            # facts guarded BY r die whenever r is written; facts ABOUT r survive a guarded clean definition (when it
            # executes the new value is clean, when it does not the old fact still applies)
            cc = {f for f in cc if f.split("?")[1].lstrip("!") != r}
            if g is None or new:
                cc = {f for f in cc if not f.startswith(r + "?")}
                for x in [x for x in t if x.startswith(r + ".b")]:
                    t.discard(x)
            if new:
                t.add(r)
            elif g is None:
                t.discard(r)
            elif r in t:
                cc.add(r + "?" + g)
                # `@P def` and `@!P def`, both from clean sources, define the register on every path
                other = r + "?" + (g[1:] if g.startswith("!") else "!" + g)
                if other in cc:
                    t.discard(r)
                    cc = {f for f in cc if not f.startswith(r + "?")}
        out = (frozenset(t), frozenset(cc))

        def resolved(lit):
            """the state on an edge along which predicate literal `lit` is known to hold: facts r?lit become plain"""
            clean = {f.split("?")[0] for f in cc if f.split("?")[1] == lit}
            return (frozenset(x for x in t if x not in clean), frozenset(cc))

        for j in succ[i]:
            edge = out
            if d["base"] == "BRA" and g is not None and d["target"] is not None and len(succ[i]) == 2:
                # `@P BRA target`: P holds on the taken edge, !P on the fall-through
                comp = g[1:] if g.startswith("!") else "!" + g
                edge = resolved(g) if j == d["target"] and j != i + 1 else resolved(comp)
            if state_in[j] is None:
                merged = edge
            else:
                # a fact about a register that is clean anyway on one side holds there vacuously
                (ta, ca), (tb, cb) = state_in[j], edge
                keep = frozenset(f for f in (ca | cb)
                                 if (f in ca or f.split("?")[0] not in ta) and (f in cb or f.split("?")[0] not in tb))
                merged = (ta | tb, keep)
            if merged != state_in[j]:
                state_in[j] = merged
                work.append(j)
    flags = []
    for i, d in enumerate(decoded):
        if state_in[i] is None:
            continue
        t, cc = state_in[i]
        g = d["guard"]
        if d["base"] in ("BRA", "EXIT", "CALL", "RET", "JMP", "BRX", "JMX", "BREAK", "KILL"):
            guards = ([g.lstrip("!")] if g else []) + d["branch_pred"] + \
                     [r for r in d["srcs"] if d["base"] in ("BRX", "JMX")]
            bad = [x for x in guards if x in t]
            if bad:
                flags.append(("secret-dependent control flow (%s)" % ",".join(bad), d))
        if d["addr_regs"]:
            bad = [r for r in d["addr_regs"] if tainted(t, cc, r, g)]
            if bad:
                flags.append(("secret-dependent address (%s)" % ",".join(bad), d))
        if d["base"].startswith(VARIABLE_TIME) and any(tainted(t, cc, r, g) for r in d["srcs"]):
            flags.append(("value-dependent latency", d))
    stats = collections.Counter(d["base"] for d in decoded)
    return flags, stats, n


def main(argv):
    jobs = []
    if len(argv) >= 2:
        jobs = [(argv[i], argv[i + 1]) for i in range(0, len(argv) - 1, 2)]
    else:
        jobs = [(os.path.join(BUILD, o), p) for o, p in DEFAULT]
    total_flags = 0
    kernels = 0
    for obj, pat in jobs:
        if not os.path.exists(obj):
            print("missing object", obj, "(run python -m modarith_b200.build)")
            return 2
        for name, ins in parse(obj, pat):
            flags, stats, n = analyse(name, ins)
            kernels += 1
            nbr = stats["BRA"] + stats["EXIT"]
            nmem = sum(v for k, v in stats.items() if k.startswith(("LD", "ST", "ATOM", "RED")) and k not in ("LDC", "LDCU"))
            short = re.sub(r"^_Z\d+", "", name)[:70]
            print("%-72s %6d instr  %3d branches/exits  %4d memory ops  -> %s" % (
                short, n, nbr, nmem, "clean" if not flags else "%d FLAGGED" % len(flags)))
            for why, d in flags[:12]:
                print("      %s: /*%04x*/ %s" % (why, d["addr"], d["text"]))
            total_flags += len(flags)
    print("%d kernels audited, %d findings" % (kernels, total_flags))
    return 1 if total_flags else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
