"""Named moduli and Montgomery-curve constants for the batched field / ladder path.

Mirrors the "user editable area" tables of the reference generators
(pseudo.py:1487-1550, monty.py:1961-2108) for the three moduli the hot path
covers, and the curve constants of rfc7748.c:120-132.  Only data lives here;
the limb plans are derived in gen/plan.py.
"""
from dataclasses import dataclass


@dataclass(frozen=True)
class Prime:
    name: str          # reference's prime name (argv[2] of pseudo.py / monty.py)
    p: int
    family: str        # "pseudo" (pseudo.py) or "monty" (monty.py) in the reference
    # Montgomery-curve constants (rfc7748.c:120-132); None for field-only moduli
    a24: int | None = None
    cof: int | None = None
    generator: int | None = None
    # short-Weierstrass curve y^2 = x^3 - 3x + b over this field (curve.py:157-166); None otherwise
    # twisted Edwards curve -x^2 + y^2 = 1 + d x^2 y^2 over this field (curve.py:85-94, ED25519); None otherwise
    ed_d: int | None = None
    ed_gx: int | None = None
    ed_gy: int | None = None
    ed_order: int | None = None
    wb: int | None = None
    wgx: int | None = None
    wgy: int | None = None
    worder: int | None = None

    @property
    def nbits(self) -> int:
        return self.p.bit_length()

    @property
    def nbytes(self) -> int:           # pseudo.py:1611-1614
        return (self.nbits + 7) // 8

    @property
    def pm1d2(self) -> int:            # pseudo.py:1574-1579: 2-adicity of p-1
        k, t = 0, self.p - 1
        while t % 2 == 0:
            k += 1
            t >>= 1
        return k

    @property
    def pe(self) -> int:               # pseudo.py:1580-1581: progenitor exponent
        e = 1 << self.pm1d2
        return (self.p - 1 - e) // (2 * e)

    @property
    def roi(self) -> int:              # pseudo.py:1616-1627: 2^k-th root of unity
        k = self.pm1d2
        p = self.p
        if k == 1:
            return p - 1
        if k == 2:
            return pow(2, (p - 1) // 4, p)
        q = 2
        while pow(q, (p - 1) // 2, p) == 1:
            q += 1
        return pow(q, (p - 1) >> k, p)


X25519 = Prime("X25519", 2**255 - 19, "pseudo", a24=121665, cof=3, generator=9,
               ed_d=0x52036CEE2B6FFE738CC740797779E89800700A4D4141D8AB75EB4DCA135978A3,
               ed_gx=0x216936D3CD6E53FEC0A4E231FDD6DC5C692CC7609525A7B2C9562D608F25D51A,
               ed_gy=0x6666666666666666666666666666666666666666666666666666666666666658,
               ed_order=0x1000000000000000000000000000000014DEF9DEA2F79CD65812631A5CF5D3ED)
X448 = Prime("X448", 2**448 - 2**224 - 1, "monty", a24=39081, cof=2, generator=5)
NIST256 = Prime("NIST256", 2**256 - 2**224 + 2**192 + 2**96 - 1, "monty",
                wb=0x5AC635D8AA3A93E7B3EBBD55769886BC651D06B0CC53B0F63BCE3C3E27D2604B,
                wgx=0x6B17D1F2E12C4247F8BCE6E563A440F277037D812DEB33A0F4A13945D898C296,
                wgy=0x4FE342E2FE1A7F9B8EE7EB4A7C0F9E162BCE33576B315ECECBB6406837BF51F5,
                worder=0xFFFFFFFF00000000FFFFFFFFFFFFFFFFBCE6FAADA7179E84F3B9CAC2FC632551)

# the three moduli of the hot path (BASELINE configs)
PRIMES = {q.name: q for q in (X25519, X448, NIST256)}

# moduli outside the hot path that are built into the library to exercise the generator's fall-back plan
# (full Montgomery, any odd modulus): a field prime that is NOT exploitable by the cheaper plans
# (monty.py:2066-2067) and a group order (the reference's "00<decimal>" mode, monty.py:2110-2127)
SECP256K1 = Prime("SECP256K1", 2**256 - 2**32 - 977, "monty")
NIST256ORDER = Prime("NIST256ORDER", 0xFFFFFFFF00000000FFFFFFFFFFFFFFFFBCE6FAADA7179E84F3B9CAC2FC632551, "monty")
EXTRA_PRIMES = {q.name: q for q in (SECP256K1, NIST256ORDER)}
ALL_PRIMES = dict(PRIMES, **EXTRA_PRIMES)

# group orders whose field code is compiled only INTO another modulus' unit (no entry points of their own, no
# mab_<NAME>_* symbols): the Ed25519 group order L, for k = SHA-512(R || A || M) mod L and the S < L check of
# Ed25519 verification (csrc/eddsa_sm100.cuh, included by mab_capi_X25519.cu)
ED25519ORDER = Prime("ED25519ORDER", 2**252 + 27742317777372353535851937790883648493, "monty")
ORDER_PRIMES = {q.name: q for q in (ED25519ORDER,)}

# Every other named modulus of the reference's tables (pseudo.py:1487-1550 "pseudo", monty.py:1961-2108 "monty"),
# as data: none of them is compiled into the shipped library, `python -m modarith_b200.build --prime NAME` builds an
# add-on library for one (libmodarith_b200_<NAME>.so, same C ABI; Field(NAME) finds it).  A name both generators
# know is listed under the family whose plan the sm_100a generator ends up choosing anyway (make_plan tries the
# plans in order of cost whatever the family says).
REFERENCE_PRIMES = {
    "PM266": ("2**266-3", "pseudo"), "NUMS256W": ("2**256-189", "pseudo"), "NUMS256E": ("2**256-189", "pseudo"),
    "NIST521": ("2**521-1", "pseudo"), "ED521": ("2**521-1", "pseudo"), "ED25519": ("2**255-19", "pseudo"),
    "C2065": ("2**206-5", "pseudo"), "PM336": ("2**336-3", "pseudo"), "PM383": ("2**383-187", "pseudo"),
    "C41417": ("2**414-17", "pseudo"), "PM512": ("2**512-569", "pseudo"),
    "NIST384": ("2**384-2**128-2**96+2**32-1", "monty"), "ED448": ("2**448-2**224-1", "monty"),
    "GM270": ("2**270-2**162-1", "monty"), "GM240": ("2**240-2**183-1", "monty"), "GM360": ("2**360-2**171-1", "monty"),
    "GM480": ("2**480-2**240-1", "monty"), "GM378": ("2**378-2**324-1", "monty"), "GM384": ("2**384-2**186-1", "monty"),
    "GM512": ("2**512-2**127-1", "monty"), "NIST224": ("2**224-2**96+1", "monty"),
    "TWEEDLE": ("0x40000000000000000000000000000000038aa127696286c9842cafd400000001", "monty"),
    "SIDH434": ("2**216*3**137-1", "monty"), "SIDH503": ("2**250*3**159-1", "monty"), "SIDH610": ("2**305*3**192-1", "monty"),
    "SIDH751": ("2**372*3**239-1", "monty"), "MFP4": ("3*67*(2**246)-1", "monty"),
    "MFP7": ("2**145*(3**9)*(59**3)*(311**3)*(317**3)*(503**3)-1", "monty"),
    "MFP1973": ("0x34e29e286b95d98c33a6a86587407437252c9e49355147ffffffffffffffffff", "monty"),
    "ED248": ("5*2**248-1", "monty"),
}


def named(name: str) -> Prime:
    """A modulus by the reference's name: one of the built-in ones, or a table entry above."""
    if name in ALL_PRIMES:
        return ALL_PRIMES[name]
    if name in REFERENCE_PRIMES:
        expr, family = REFERENCE_PRIMES[name]
        return Prime(name, eval(expr, {"__builtins__": {}}), family)
    raise KeyError(name)
