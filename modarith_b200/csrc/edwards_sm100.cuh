// edwards_sm100.cuh -- twisted Edwards group law (a = -1: Ed25519) on the batched field, one point per
// thread.  Counterpart of edwards.c: standard projective addition and doubling from the EFD
// (add-2008-bbjlp / dbl-2008-bbjlp, which edwards.c:73-145 also transcribes; complete for Ed25519
// because d is a non-square), point set with the on-curve check (edwards.c:243-272,347-356), affine/get
// (edwards.c:184-241).  The identity is (0:1:1) and is reported as (0, 1).
#pragma once
#include "mab_field.cuh"
#include "ecnmul_sm100.cuh"

template <class F> struct Edwards {
  static constexpr int L = F::L;
  typedef Field<F> Fd;
  struct Pt { uint32_t x[L], y[L], z[L]; };
  // k_ecnmul: where the fixed-window table lives and how many CTAs per SM the registers are cut for (measured)
  static constexpr bool ECN_GLOBAL_TABLE = false;
  static constexpr int ECN_MINBLOCKS = 2;
  static constexpr int ECN2_MINBLOCKS = 2;

  static MAB_DEV void inf(Pt& P) { Fd::zer(P.x); Fd::one(P.y); Fd::one(P.z); }           // edwards.c:170-175
  static MAB_DEV void cpy(Pt& R, const Pt& P) { Fd::cpy(R.x, P.x); Fd::cpy(R.y, P.y); Fd::cpy(R.z, P.z); }
  static MAB_DEV void cmv(uint32_t d, const Pt& Q, Pt& P) { Fd::cmv(d, Q.x, P.x); Fd::cmv(d, Q.y, P.y); Fd::cmv(d, Q.z, P.z); }
  static MAB_DEV void neg(Pt& P) { uint32_t t[L]; F::neg(t, P.x); Fd::cpy(P.x, t); }     // edwards.c:66-69

  // P <- P + Q  (a = -1): 10M + 1S + 1 mul-by-d
  struct Seq {};                                   // no ordering needed on this field (see Weierstrass::Seq)
  static MAB_DEV Seq seq(uint32_t) { return Seq(); }
  static MAB_DEV void add(Pt& P, const Pt& Q, Seq&) { add(P, Q); }
  static MAB_DEV void dbl(Pt& P, Seq&) { dbl(P); }
  static MAB_DEV void dbl4(Pt& P, Seq&) { dbl(P); dbl(P); dbl(P); dbl(P); }
  template <int N> static MAB_DEV void dbln(Pt& P, Seq&) {
    for (int i = 0; i < N; i++) dbl(P);
  }
  // e*P + f*Q with joint 2-bit windows (EcnMul::mul2w; the 16-entry table lives in the global workspace)
#ifndef MAB_ED_MUL2_WINDOW
#define MAB_ED_MUL2_WINDOW 1
#endif
  static constexpr bool MUL2_WINDOW = (MAB_ED_MUL2_WINDOW != 0);
  static MAB_DEV void add(Pt& P, const Pt& Q) {
    uint32_t A[L], B[L], C[L], D[L], E[L], Ff[L], Gg[L], dd[L];
    F::set_ed_d(dd);
    F::mul(A, P.z, Q.z);
    F::sqr(B, A);
    F::mul(C, P.x, Q.x);
    F::mul(D, P.y, Q.y);
    F::mul(E, C, D);
    F::mul(E, E, dd);
    F::sub_tt(Ff, B, E);
    F::add_tt(Gg, B, E);
    F::add_tt(B, P.x, P.y);
    F::add(E, Q.x, Q.y);                         // Q is not necessarily a product: general form
    F::mul(B, B, E);
    F::sub_tt(B, B, C);
    F::sub(B, B, D);                             // B is a difference by now: general form
    F::mul(B, B, Ff);
    F::mul(P.x, B, A);                           // X3 = A*F*((X1+Y1)(X2+Y2)-C-D)
    F::add_tt(D, D, C);                          // D - a*C with a = -1
    F::mul(D, D, A);
    F::mul(P.y, D, Gg);                          // Y3 = A*G*(D+C)
    F::mul(P.z, Ff, Gg);                         // Z3 = F*G
  }

  // P <- 2P  (a = -1): 3M + 4S
  static MAB_DEV void dbl(Pt& P) {
    uint32_t B[L], C[L], D[L], H[L], Ff[L], J[L];
    F::add_tt(B, P.x, P.y);
    F::sqr(B, B);
    F::sqr(C, P.x);
    F::sqr(D, P.y);
    F::sqr(H, P.z);
    F::add_tt(H, H, H);
    F::sub_tt(Ff, D, C);                         // F = a*C + D = D - C
    F::sub(J, Ff, H);                            // J = F - 2Z^2
    F::sub_tt(B, B, C);
    F::sub(B, B, D);
    F::mul(P.x, B, J);                           // X3 = (B-C-D)*J
    F::add_tt(C, C, D);
    F::neg(C, C);                                // E - D = -C - D
    F::mul(P.y, Ff, C);                          // Y3 = F*(E-D)
    F::mul(P.z, Ff, J);                          // Z3 = F*J
  }

  // ecnXXXset with both coordinates (edwards.c:243-272): (x,y) if -x^2 + y^2 = 1 + d x^2 y^2, else identity
  static MAB_DEV void set(Pt& P, const uint32_t (&xw)[L], const uint32_t (&yw)[L]) {
    uint32_t X[L], Y[L], U[L], V[L], dd[L], one[L];
    (void)Fd::from_words(P.x, xw);
    (void)Fd::from_words(P.y, yw);
    F::sqr(X, P.x);
    F::sqr(Y, P.y);
    F::sub(U, Y, X);
    F::mul(V, X, Y);
    F::set_ed_d(dd);
    F::mul(V, V, dd);
    Fd::one(one);
    F::add(V, V, one);
    const uint32_t bad = 1u - Fd::cmp(U, V);
    if (F::TIGHT) {                                // imported words may be anything below 2^(32L): x*1, y*1 are products
      F::mul(P.x, P.x, one);
      F::mul(P.y, P.y, one);
    }
    Fd::one(P.z);
    Pt O;
    inf(O);
    cmv(bad, O, P);
  }

  // ecnXXXget (edwards.c:184-241): affine coordinates as canonical plain words; z = 0 -> (0, 1)
  static MAB_DEV void get(uint32_t (&xw)[L], uint32_t (&yw)[L], const Pt& P) {
    uint32_t i[L], x[L], y[L], one[L];
    Fd::template inv<false>(i, P.z, P.z);
    F::mul(x, P.x, i);
    F::mul(y, P.y, i);
    Fd::one(one);
    Fd::cmv(Fd::is0_stored(P.z), one, y);
    Fd::to_words(xw, x);
    Fd::to_words(yw, y);
  }

  // Point decoding of RFC 8032 section 5.1.3, strict: enc = y (low 255 bits) | sign of x << 255, little-endian
  // words.  1 iff y < p, x^2 = (y^2 - 1) / (d y^2 + 1) has a root and not (x = 0 with the sign bit set); P is the
  // point (coordinates tight, as set() leaves them) where ok = 1 and O elsewhere.  One progenitor chain:
  // x = u v^3 (u v^7)^((p-5)/8), then x *= sqrt(-1) where v x^2 = -u (p = 5 mod 8).  Every check is a mask.
  static MAB_DEV uint32_t decode(Pt& P, const uint32_t (&enc)[L]) {
    static_assert(F::PM1D2 == 2, "the (p-5)/8 square-root chain needs p = 5 mod 8");
    uint32_t yw[L], y[L], u[L], v[L], t[L], x[L], w[L], one[L];
#pragma unroll
    for (int j = 0; j < L; j++) yw[j] = enc[j];
    const uint32_t sgn = yw[L - 1] >> 31;
    yw[L - 1] &= 0x7fffffffu;
    uint32_t ok = Fd::from_words(y, yw);
    Fd::one(one);
    F::sqr(u, y);
    F::set_ed_d(t);
    F::mul(v, u, t);
    F::add(v, v, one);                             // v = d y^2 + 1 (never 0: d is a non-square)
    F::sub(u, u, one);                             // u = y^2 - 1
    F::sqr(t, v);
    F::mul(t, t, v);                               // v^3
    F::mul(x, u, t);                               // u v^3
    F::sqr(t, t);
    F::mul(t, t, v);                               // v^7
    F::mul(t, t, u);                               // u v^7
    F::pro(w, t);                                  // (u v^7)^((p-5)/8)
    F::mul(x, x, w);
    F::sqr(t, x);
    F::mul(t, t, v);                               // v x^2
    const uint32_t is_u = Fd::cmp(t, u);
    F::neg(w, u);
    const uint32_t is_neg_u = Fd::cmp(t, w);
    F::set_roi(w);
    F::mul(t, x, w);
    Fd::cmv(is_neg_u, t, x);
    ok &= is_u | is_neg_u;
    uint32_t xc[L];
    Fd::to_words(xc, x);
    uint32_t nz = 0;
#pragma unroll
    for (int j = 0; j < L; j++) nz |= xc[j];
    ok &= 1u - (sgn & (nz == 0 ? 1u : 0u));
    F::neg(t, x);
    Fd::cmv((xc[0] & 1u) ^ sgn, t, x);
    F::mul(P.x, x, one);                           // products: tight whatever neg / import left
    F::mul(P.y, y, one);
    Fd::one(P.z);
    Pt O;
    inf(O);
    cmv(1u - ok, O, P);
    return ok;
  }

  // Point encoding (RFC 8032 section 5.1.2): canonical y with the low bit of x in bit 255, little-endian words.
  // One inversion of Z (Z != 0 for every point the complete formulas produce).
  static MAB_DEV void encode(uint32_t (&enc)[L], const Pt& P) {
    uint32_t i[L], x[L], y[L], xw[L];
    Fd::template inv<false>(i, P.z, P.z);
    F::mul(x, P.x, i);
    F::mul(y, P.y, i);
    Fd::to_words(xw, x);
    Fd::to_words(enc, y);
    enc[L - 1] |= xw[0] << 31;
  }
};
