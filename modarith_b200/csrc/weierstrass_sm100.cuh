// weierstrass_sm100.cuh -- short-Weierstrass group law (A = -3) and constant-time scalar multiplication
// on the batched field, one point per thread.  SURVEY.md section 8(f) row 1: the direct consumer of the
// P-256 field work.
//
// Counterpart of weierstrass.c: complete projective addition and doubling from eprint 2015/1060
// (Renes, Costello, Batina; Algorithms 4 and 6 for a = -3, which weierstrass.c:69-176,187-282 also
// transcribes), point set/validate (weierstrass.c:364-427), affine/get (:297-349) and the fixed-window
// signed-digit multiplication ecnXXXmul (:441-542): table O,P,..,8P, nibbles recoded to digits in
// [-8,7], every lookup a scan of the whole table with masks.  Results are compared as affine (x,y) byte
// strings, which are unique, so only the values -- not the order of internal operations -- are pinned.
#pragma once
#include "mab_field.cuh"
#include "ecnmul_sm100.cuh"

template <class F> struct Weierstrass {
  static constexpr int L = F::L;
  typedef Field<F> Fd;
  struct Pt { uint32_t x[L], y[L], z[L]; };
  // k_ecnmul: where the fixed-window table lives and how many CTAs per SM the registers are cut for (measured,
  // profiles/r2_ecn_variants.txt).  Round 1 ran three CTAs at 168 registers (700 bytes of spill) with the table in
  // a global workspace; with the Jacobian doubling runs the loop needs the registers more than the warps: two CTAs
  // at 255 registers with the nine-entry table in shared memory (2 x 108 KB) give 21.6 M/s against 17.6 / 18.8
  // (three CTAs / two CTAs with the global table).  k_ecnmul2 (sixteen-entry table, always global) stays at three.
  static constexpr bool ECN_GLOBAL_TABLE = false;
  static constexpr int ECN_MINBLOCKS = 2;
  static constexpr int ECN2_MINBLOCKS = 3;

  static MAB_DEV void inf(Pt& P) { Fd::zer(P.x); Fd::one(P.y); Fd::zer(P.z); }          // weierstrass.c:283-288
  static MAB_DEV void cpy(Pt& R, const Pt& P) { Fd::cpy(R.x, P.x); Fd::cpy(R.y, P.y); Fd::cpy(R.z, P.z); }
  static MAB_DEV void cmv(uint32_t d, const Pt& Q, Pt& P) { Fd::cmv(d, Q.x, P.x); Fd::cmv(d, Q.y, P.y); Fd::cmv(d, Q.z, P.z); }

  // Ordering of the multiplications inside add/dbl.  The formulas offer ptxas up to three independent
  // multiplications at a time; it interleaves them all, and with the carry chains of the Montgomery
  // reduction that needs more predicate registers than exist (measured: ~1200 of 15000 instructions per
  // digit were predicate saves and restores).  Seq makes every multiplication's first operand word
  // depend on the result of the one DEPTH multiplications earlier through `x ^ (r & z)` with a zero z
  // that the compiler cannot see (one LOP3 per multiplication), which bounds the overlap to DEPTH.
#ifndef MAB_ECN_CHAIN
#define MAB_ECN_CHAIN 2
#endif
  struct Seq {
    uint32_t z, l0, l1;
    MAB_DEV void done(uint32_t w) {
      if (MAB_ECN_CHAIN == 1) l0 = w;
      else { l0 = l1; l1 = w; }
    }
  };
  static MAB_DEV void mulq(Seq& q, uint32_t (&r)[L], const uint32_t (&a)[L], const uint32_t (&b)[L]) {
    if (MAB_ECN_CHAIN == 0) { F::mul(r, a, b); return; }
    uint32_t a2[L];
    Fd::cpy(a2, a);
    a2[0] ^= q.l0 & q.z;
    F::mul(r, a2, b);
    q.done(r[L - 1]);
  }
  static MAB_DEV void sqrq(Seq& q, uint32_t (&r)[L], const uint32_t (&a)[L]) {
    if (MAB_ECN_CHAIN == 0) { F::sqr(r, a); return; }
    uint32_t a2[L];
    Fd::cpy(a2, a);
    a2[0] ^= q.l0 & q.z;
    F::sqr(r, a2);
    q.done(r[L - 1]);
  }

  // P <- P + Q, complete (eprint 2015/1060 Algorithm 4, a = -3): 12M + 2 mul-by-b + 29 add/sub
  static MAB_DEV Seq seq(uint32_t z) { Seq q = {z, 0, 0}; return q; }
  static MAB_DEV void add(Pt& P, const Pt& Q) { Seq q = seq(0); add(P, Q, q); }
  static MAB_DEV void dbl(Pt& P) { Seq q = seq(0); dbl(P, q); }
  static MAB_DEV void add(Pt& P, const Pt& Q, Seq& q) {
    uint32_t b[L], t0[L], t1[L], t2[L], t3[L], t4[L], x3[L], y3[L], z3[L];
    F::set_b(b);
    mulq(q, t0, P.x, Q.x);  mulq(q, t1, P.y, Q.y);  mulq(q, t2, P.z, Q.z);
    F::add(t3, P.x, P.y);  F::add(t4, Q.x, Q.y);  mulq(q, t3, t3, t4);
    F::add(t4, t0, t1);    F::sub(t3, t3, t4);    F::add(t4, P.y, P.z);
    F::add(x3, Q.y, Q.z);  mulq(q, t4, t4, x3);    F::add(x3, t1, t2);
    F::sub(t4, t4, x3);    F::add(x3, P.x, P.z);  F::add(y3, Q.x, Q.z);
    mulq(q, x3, x3, y3);    F::add(y3, t0, t2);    F::sub(y3, x3, y3);
    mulq(q, z3, b, t2);     F::sub(x3, y3, z3);    F::add(z3, x3, x3);
    F::add(x3, x3, z3);    F::sub(z3, t1, x3);    F::add(x3, t1, x3);
    mulq(q, y3, b, y3);     F::add(t1, t2, t2);    F::add(t2, t1, t2);
    F::sub(y3, y3, t2);    F::sub(y3, y3, t0);    F::add(t1, y3, y3);
    F::add(y3, t1, y3);    F::add(t1, t0, t0);    F::add(t0, t1, t0);
    F::sub(t0, t0, t2);    mulq(q, t1, t4, y3);    mulq(q, t2, t0, y3);
    mulq(q, y3, x3, z3);    F::add(y3, y3, t2);    mulq(q, x3, t3, x3);
    F::sub(x3, x3, t1);    mulq(q, z3, t4, z3);    mulq(q, t1, t3, t0);
    F::add(z3, z3, t1);
    Fd::cpy(P.x, x3); Fd::cpy(P.y, y3); Fd::cpy(P.z, z3);
  }

  // P <- 2P, complete (Algorithm 6, a = -3): 8M + 3S + 2 mul-by-b + 21 add/sub
  static MAB_DEV void dbl(Pt& P, Seq& q) {
    uint32_t b[L], t0[L], t1[L], t2[L], t3[L], x3[L], y3[L], z3[L];
    F::set_b(b);
    sqrq(q, t0, P.x);       sqrq(q, t1, P.y);       sqrq(q, t2, P.z);
    mulq(q, t3, P.x, P.y);  F::add(t3, t3, t3);    mulq(q, z3, P.x, P.z);
    F::add(z3, z3, z3);    mulq(q, y3, b, t2);     F::sub(y3, y3, z3);
    F::add(x3, y3, y3);    F::add(y3, x3, y3);    F::sub(x3, t1, y3);
    F::add(y3, t1, y3);    mulq(q, y3, x3, y3);    mulq(q, x3, x3, t3);
    F::add(t3, t2, t2);    F::add(t2, t2, t3);    mulq(q, z3, b, z3);
    F::sub(z3, z3, t2);    F::sub(z3, z3, t0);    F::add(t3, z3, z3);
    F::add(z3, z3, t3);    F::add(t3, t0, t0);    F::add(t0, t3, t0);
    F::sub(t0, t0, t2);    mulq(q, t0, t0, z3);    F::add(y3, y3, t0);
    mulq(q, t0, P.y, P.z);  F::add(t0, t0, t0);    mulq(q, z3, t0, z3);
    F::sub(x3, x3, z3);    mulq(q, z3, t0, t1);    F::add(z3, z3, z3);
    F::add(z3, z3, z3);
    Fd::cpy(P.x, x3); Fd::cpy(P.y, y3); Fd::cpy(P.z, z3);
  }

  // P <- 2^N P: the four doublings between two digits of the window method (weierstrass.c:528-531 calls ecnXXXdbl
  // four times), the two between joint digits of e*P + f*Q.  The complete doubling above is 8M + 3S + 2 multiplications by b = 13 products; on a curve of prime
  // order with a = -3 the Jacobian doubling (delta = Z^2, gamma = Y^2, beta = X gamma, alpha = 3 (X - delta)(X + delta),
  // X' = alpha^2 - 8 beta, Z' = (Y + Z)^2 - gamma - delta, Y' = alpha (4 beta - X') - 8 gamma^2: 3M + 5S) is valid
  // for EVERY point -- there is no point of order two, and infinity (Z = 0) stays at Z' = 0 -- so the run of four is
  // done there: homogeneous (X : Y : Z) -> Jacobian (X Z : Y Z^2 : Z) costs 2M + 1S, back (X' Z' : Y' : Z'^3) 2M + 1S,
  // 36 products instead of 52 (the squaring of Z is shared between consecutive doublings and the changes of coordinates), 16 fewer field additions.  The only repair: infinity comes back as (0 : 0 : 0), which
  // the complete addition would not recognise; Y is set to 1 wherever Z is 0.  The affine result, which is what the
  // reference's outputs pin, is the same; MAB_ECN_JACOBIAN=0 keeps the four complete doublings (comparison builds).
#ifndef MAB_ECN_JACOBIAN
#define MAB_ECN_JACOBIAN 1
#endif
  static MAB_DEV void dbl4(Pt& P, Seq& q) { dbln<4>(P, q); }
  // e*P + f*Q is done with joint 2-bit windows (EcnMul::mul2w): a 16-entry table in the global workspace
  static constexpr bool MUL2_WINDOW = true;
  template <int N> static MAB_DEV void dbln(Pt& P, Seq& q) {
    if (!MAB_ECN_JACOBIAN) {
      for (int i = 0; i < N; i++) dbl(P, q);
      return;
    }
    uint32_t X[L], Y[L], Z[L], d[L], g[L], b[L], a[L], t[L];
    sqrq(q, d, P.z);                               // delta = Z^2, also what the change of coordinates needs
    mulq(q, X, P.x, P.z);                          // X Z
    mulq(q, Y, P.y, d);                            // Y Z^2
    Fd::cpy(Z, P.z);
    // Halved form of the doubling: with L = alpha/2 the point (X'/4 : Y'/8 : Z'/2) -- the same point -- is
    //   X'' = L^2 - 2 beta,  Y'' = L (beta - X'') - gamma^2,  Z'' = Y Z,
    // 4M + 4S like the textbook form but 9 field additions / subtractions and one halving instead of 16 (the
    // multiples 4 beta, 8 beta, 8 gamma^2 are gone); on this field an addition costs a quarter of a product.
    static_assert(F::MONTGOMERY, "haf_reduced below relies on fully reduced stored values");
    MAB_NOUNROLL
    for (int i = 0; i < N; i++) {
      sqrq(q, g, Y);                               // gamma
      mulq(q, b, X, g);                            // beta
      F::sub(t, X, d);  F::add(a, X, d);
      mulq(q, a, a, t);                            // (X - delta)(X + delta)
      F::add(t, a, a);  F::add(a, a, t);           // alpha = 3 (..)
      Fd::haf_reduced(a);                          // L = alpha / 2
      mulq(q, Z, Y, Z);                            // Z'' = Y Z
      sqrq(q, X, a);
      F::sub(X, X, b);  F::sub(X, X, b);           // X'' = L^2 - 2 beta
      F::sub(t, b, X);                             // beta - X''
      mulq(q, t, a, t);
      sqrq(q, g, g);                               // gamma^2
      F::sub(Y, t, g);                             // Y'' = L (beta - X'') - gamma^2
      sqrq(q, d, Z);                               // delta of the next doubling / Z^2 for the way back
    }
    mulq(q, P.x, X, Z);                            // X Z
    mulq(q, P.z, d, Z);                            // Z^3
    uint32_t one[L];
    Fd::one(one);
    Fd::cmv(Fd::is0_stored(P.z), one, Y);          // infinity: (0 : 1 : 0)
    Fd::cpy(P.y, Y);
  }

  // ecnXXXset with both coordinates (weierstrass.c:364-396,415-427): (x,y) if y^2 = x^3 - 3x + b, else O.
  // xw, yw: plain values as little-endian words (any value < 2^(32L): modimp semantics)
  static MAB_DEV void set(Pt& P, const uint32_t (&xw)[L], const uint32_t (&yw)[L]) {
    uint32_t v[L], t[L], b[L];
    (void)Fd::from_words(P.x, xw);
    (void)Fd::from_words(P.y, yw);
    F::sqr(v, P.x);
    F::mul(v, v, P.x);
    F::sub(v, v, P.x); F::sub(v, v, P.x); F::sub(v, v, P.x);
    F::set_b(b);
    F::add(v, v, b);
    F::sqr(t, P.y);
    const uint32_t bad = 1u - Fd::cmp(t, v);
    Fd::one(P.z);
    Pt O;
    inf(O);
    cmv(bad, O, P);
  }
  // set() that reports what it checked: 1 iff xw < p, yw < p and (x, y) is on the curve (public-key validation,
  // SEC1 v2 section 3.2.2.1); P is O otherwise.  set() keeps modimp semantics (a coordinate >= p reduces).
  static MAB_DEV uint32_t set_checked(Pt& P, const uint32_t (&xw)[L], const uint32_t (&yw)[L]) {
    uint32_t v[L], t[L], b[L];
    const uint32_t lt = Fd::from_words(P.x, xw) & Fd::from_words(P.y, yw);
    F::sqr(v, P.x);
    F::mul(v, v, P.x);
    F::sub(v, v, P.x); F::sub(v, v, P.x); F::sub(v, v, P.x);
    F::set_b(b);
    F::add(v, v, b);
    F::sqr(t, P.y);
    const uint32_t on = Fd::cmp(t, v);
    Fd::one(P.z);
    Pt O;
    inf(O);
    cmv(1u - on, O, P);
    return lt & on;
  }

  // ecnXXXget (weierstrass.c:297-349): affine coordinates as canonical plain words; O -> (0, 1)
  static MAB_DEV void get(uint32_t (&xw)[L], uint32_t (&yw)[L], const Pt& P) {
    uint32_t i[L], x[L], y[L], one[L];
    Fd::template inv<false>(i, P.z, P.z);          // 0 -> 0
    F::mul(x, P.x, i);
    F::mul(y, P.y, i);
    Fd::one(one);
    Fd::cmv(Fd::is0_stored(P.z), one, y);
    Fd::to_words(xw, x);
    Fd::to_words(yw, y);
  }

  static MAB_DEV void neg(Pt& P) { uint32_t t[L]; F::neg(t, P.y); Fd::cpy(P.y, t); }    // weierstrass.c:62-65
};
