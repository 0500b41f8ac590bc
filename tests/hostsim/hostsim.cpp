// tests/hostsim/hostsim.cpp -- TEST SCAFFOLDING ONLY (never part of the shipped library).
//
// Compiles the GENERATED field headers and the hand-written device templates
// (mab_field.cuh, rfc7748_sm100.cuh) for the host with -DMAB_HOSTSIM, where every inline-PTX
// block is replaced by its plain-C transcription (gen/ptx.py emit_sim).  The CPU test-suite
// uses it to check the device-side logic against the oracle where there is no GPU; the GPU
// tests then check the real PTX build through the C ABI.
#define MAB_HOSTSIM 1
#include <string.h>
#include "gen/field_X25519.cuh"
#include "gen/field_X448.cuh"
#include "gen/field_NIST256.cuh"
#include "gen/field_SECP256K1.cuh"
#include "gen/field_NIST256ORDER.cuh"
#include "rfc7748_sm100.cuh"
#include "weierstrass_sm100.cuh"
#include "edwards_sm100.cuh"

enum SimOp {
  S_ADD, S_SUB, S_NEG, S_MUL, S_SQR, S_MLI, S_NSQR, S_PRO, S_INV, S_INVH, S_QR, S_QRH, S_SQRT, S_SQRTH,
  S_IS1, S_IS0, S_ONE, S_INT, S_NRES, S_REDC, S_CSW, S_CMV, S_SHL, S_SHR, S_HAF, S_2R, S_SIGN, S_CMP, S_FSB,
  S_IMPW, S_EXPW,
  // the generated blocks on their own, on any stored words (tests/test_gpu_blocks.py)
  S_MLA, S_ADDTT, S_SUBTT, S_MULW, S_SQRW, S_CANON, S_REDCW
};

template <class F> static int sim_op(int op, const uint32_t* pa, const uint32_t* pb, uint32_t scalar, uint32_t* pr, uint32_t* pr2) {
  constexpr int L = F::L;
  typedef Field<F> Fd;
  uint32_t a[L], b[L], r[L];
  for (int i = 0; i < L; i++) { a[i] = pa ? pa[i] : 0; b[i] = pb ? pb[i] : 0; r[i] = 0; }
  int ret = 0;
  switch (op) {
    case S_ADD: F::add(r, a, b); break;
    case S_SUB: F::sub(r, a, b); break;
    case S_NEG: F::neg(r, a); break;
    case S_MUL: F::mul(r, a, b); break;
    case S_SQR: F::sqr(r, a); break;
    case S_MLI: F::mli(r, a, scalar); break;
    case S_NSQR: Fd::cpy(r, a); Fd::nsqr(r, (int)scalar); break;
    case S_PRO: F::pro(r, a); break;
    case S_INV: Fd::template inv<false>(r, a, a); break;
    case S_INVH: Fd::template inv<true>(r, a, b); break;
    case S_QR: ret = (int)Fd::template qr<false>(a, a); break;
    case S_QRH: ret = (int)Fd::template qr<true>(a, b); break;
    case S_SQRT: Fd::template sqrt<false>(r, a, a); break;
    case S_SQRTH: Fd::template sqrt<true>(r, a, b); break;
    case S_IS1: ret = (int)Fd::is1(a); break;
    case S_IS0: ret = (int)Fd::is0(a); break;
    case S_ONE: Fd::one(r); break;
    case S_INT: Fd::from_int(r, scalar); break;
    case S_NRES: F::nres(r, a); break;
    case S_REDC: Fd::to_words(r, a); break;
    case S_CSW: Fd::csw(scalar & 1u, a, b); Fd::cpy(r, a); for (int i = 0; i < L; i++) pr2[i] = b[i]; break;
    case S_CMV: Fd::cmv(scalar & 1u, a, b); Fd::cpy(r, b); break;
    case S_SHL: Fd::cpy(r, a); Fd::shl(r, scalar); break;
    case S_SHR: Fd::cpy(r, a); ret = (int)Fd::shr(r, scalar); break;
    case S_HAF: Fd::cpy(r, a); Fd::haf(r); break;
    case S_2R: Fd::pow2(r, scalar); break;
    case S_SIGN: ret = (int)Fd::sign(a); break;
    case S_CMP: ret = (int)Fd::cmp(a, b); break;
    case S_FSB: Fd::cpy(r, a); ret = (int)Fd::fsb(r); break;
    case S_IMPW: ret = (int)Fd::from_words(r, a); break;
    case S_EXPW: Fd::to_words(r, a); break;
    case S_MLA: F::mla(r, a, scalar, b); break;
    case S_ADDTT: F::add_tt(r, a, b); break;
    case S_SUBTT: F::sub_tt(r, a, b); break;
    case S_MULW: F::mul_w(r, a, b); break;
    case S_SQRW: F::sqr_w(r, a); break;
    case S_CANON: ret = (int)F::canon(r, a); break;
    case S_REDCW: F::redc(r, a); break;
    default: return -1;
  }
  for (int i = 0; i < L; i++) pr[i] = r[i];
  return ret;
}

template <class F, bool VALIDATE = false> static void sim_rfc7748(const unsigned char* bk, const unsigned char* bu, unsigned char* bv) {
  constexpr int L = F::L;
  uint32_t k[L], u[L], out[L];
  memcpy(k, bk, 4 * L);
  memcpy(u, bu, 4 * L);
  if (F::LADDER_STASH) {
    uint32_t stash[2 * L];                       // stands in for the per-thread shared-memory column
    Rfc7748<F>::template scalarmult<VALIDATE>(out, k, u, stash, 1);
  } else {
    Rfc7748<F>::template scalarmult<VALIDATE>(out, k, u);
  }
  memcpy(bv, out, 4 * L);
}

// K keys through one simulated thread: K ladders, then Rfc7748<F>::finish_batch (one shared inversion)
template <class F> static void sim_rfc7748_shared_inversion(const unsigned char* bk, const unsigned char* bu, unsigned char* bv, int K) {
  constexpr int L = F::L;
  uint32_t st[4 * 3 * L];
  uint32_t stash[2 * L];
  for (int j = 0; j < K; j++) {
    uint32_t k[L], u[L], x1[L], x2[L], z2[L];
    memcpy(k, bk + 4 * L * j, 4 * L);
    memcpy(u, bu + 4 * L * j, 4 * L);
    Rfc7748<F>::ladder(x2, z2, x1, k, u, F::LADDER_STASH ? stash : nullptr, 1);
    Rfc7748<F>::st_(st, 1, j, 0, x2);
    Rfc7748<F>::st_(st, 1, j, 1, z2);
  }
  Rfc7748<F>::finish_batch(st, 1, K);
  for (int j = 0; j < K; j++) {
    uint32_t out[L];
    Rfc7748<F>::ld(out, st, 1, j, 0);
    memcpy(bv + 4 * L * j, out, 4 * L);
  }
}

// ecnXXXset + ecnXXXmul + ecnXXXget on big-endian byte strings, table in a local array
template <class F, class G> static void sim_ecnmul(const unsigned char* e, const unsigned char* x, const unsigned char* y,
                                          unsigned char* xo, unsigned char* yo) {
  constexpr int L = F::L;
  uint32_t ew[L], xw[L], yw[L];
  for (int j = 0; j < L; j++) { ew[j] = xw[j] = yw[j] = 0; }
  for (int b = 0; b < 4 * L; b++) {
    int pos = 4 * L - 1 - b;
    ew[pos >> 2] |= (uint32_t)e[b] << (8 * (pos & 3));
    xw[pos >> 2] |= (uint32_t)x[b] << (8 * (pos & 3));
    yw[pos >> 2] |= (uint32_t)y[b] << (8 * (pos & 3));
  }
  static uint4 tab[9 * 3 * L / 4];
  static uint32_t scr[2 * L];
  typename G::Pt P;
  G::set(P, xw, yw);
  // odd scalars take the register path for the digits, even ones the scratch column the kernel uses
  EcnMul<G>::mul(P, ew, tab, 1, (ew[0] & 1u) ? nullptr : scr);
  G::get(xw, yw, P);
  for (int b = 0; b < 4 * L; b++) {
    int pos = 4 * L - 1 - b;
    xo[b] = (unsigned char)(xw[pos >> 2] >> (8 * (pos & 3)));
    yo[b] = (unsigned char)(yw[pos >> 2] >> (8 * (pos & 3)));
  }
}

// ecnXXXset x2 + ecnXXXmul2 + ecnXXXget
template <class F, class G> static void sim_ecnmul2(const unsigned char* e, const unsigned char* x1, const unsigned char* y1,
                                           const unsigned char* f, const unsigned char* x2, const unsigned char* y2,
                                           unsigned char* xo, unsigned char* yo) {
  constexpr int L = F::L;
  uint32_t w[6][L];
  const unsigned char* src[6] = {e, x1, y1, f, x2, y2};
  for (int k = 0; k < 6; k++) {
    for (int j = 0; j < L; j++) w[k][j] = 0;
    for (int b = 0; b < 4 * L; b++) {
      int pos = 4 * L - 1 - b;
      w[k][pos >> 2] |= (uint32_t)src[k][b] << (8 * (pos & 3));
    }
  }
  static uint4 tab[16 * 3 * L / 4];
  static uint32_t scr[4 * (L + 1)];
  typename G::Pt P, Q, R;
  G::set(P, w[1], w[2]);
  G::set(Q, w[4], w[5]);
  if (G::MUL2_WINDOW) EcnMul<G>::mul2w(R, w[0], P, w[3], Q, tab, 1, scr);
  else EcnMul<G>::mul2(R, w[0], P, w[3], Q, tab, 1, scr);
  uint32_t xw[L], yw[L];
  G::get(xw, yw, R);
  for (int b = 0; b < 4 * L; b++) {
    int pos = 4 * L - 1 - b;
    xo[b] = (unsigned char)(xw[pos >> 2] >> (8 * (pos & 3)));
    yo[b] = (unsigned char)(yw[pos >> 2] >> (8 * (pos & 3)));
  }
}

extern "C" {
void sim_NIST256_ecnmul2(const unsigned char* e, const unsigned char* x1, const unsigned char* y1, const unsigned char* f, const unsigned char* x2, const unsigned char* y2, unsigned char* xo, unsigned char* yo) { sim_ecnmul2<F_NIST256, Weierstrass<F_NIST256> >(e, x1, y1, f, x2, y2, xo, yo); }
void sim_ED25519_ecnmul2(const unsigned char* e, const unsigned char* x1, const unsigned char* y1, const unsigned char* f, const unsigned char* x2, const unsigned char* y2, unsigned char* xo, unsigned char* yo) { sim_ecnmul2<F_X25519, Edwards<F_X25519> >(e, x1, y1, f, x2, y2, xo, yo); }
void sim_NIST256_ecnmul(const unsigned char* e, const unsigned char* x, const unsigned char* y, unsigned char* xo, unsigned char* yo) { sim_ecnmul<F_NIST256, Weierstrass<F_NIST256> >(e, x, y, xo, yo); }
void sim_ED25519_ecnmul(const unsigned char* e, const unsigned char* x, const unsigned char* y, unsigned char* xo, unsigned char* yo) { sim_ecnmul<F_X25519, Edwards<F_X25519> >(e, x, y, xo, yo); }
void sim_X25519_rfc7748_shared(const unsigned char* bk, const unsigned char* bu, unsigned char* bv, int K) { sim_rfc7748_shared_inversion<F_X25519>(bk, bu, bv, K); }
void sim_X448_rfc7748_shared(const unsigned char* bk, const unsigned char* bu, unsigned char* bv, int K) { sim_rfc7748_shared_inversion<F_X448>(bk, bu, bv, K); }
int sim_X25519_op(int op, const uint32_t* a, const uint32_t* b, uint32_t s, uint32_t* r, uint32_t* r2) { return sim_op<F_X25519>(op, a, b, s, r, r2); }
int sim_X448_op(int op, const uint32_t* a, const uint32_t* b, uint32_t s, uint32_t* r, uint32_t* r2) { return sim_op<F_X448>(op, a, b, s, r, r2); }
int sim_NIST256_op(int op, const uint32_t* a, const uint32_t* b, uint32_t s, uint32_t* r, uint32_t* r2) { return sim_op<F_NIST256>(op, a, b, s, r, r2); }
int sim_SECP256K1_op(int op, const uint32_t* a, const uint32_t* b, uint32_t s, uint32_t* r, uint32_t* r2) { return sim_op<F_SECP256K1>(op, a, b, s, r, r2); }
int sim_NIST256ORDER_op(int op, const uint32_t* a, const uint32_t* b, uint32_t s, uint32_t* r, uint32_t* r2) { return sim_op<F_NIST256ORDER>(op, a, b, s, r, r2); }
void sim_X25519_rfc7748(const unsigned char* bk, const unsigned char* bu, unsigned char* bv) { sim_rfc7748<F_X25519>(bk, bu, bv); }
void sim_X448_rfc7748(const unsigned char* bk, const unsigned char* bu, unsigned char* bv) { sim_rfc7748<F_X448>(bk, bu, bv); }
void sim_X25519_rfc7748_validate(const unsigned char* bk, const unsigned char* bu, unsigned char* bv) { sim_rfc7748<F_X25519, true>(bk, bu, bv); }
void sim_X448_rfc7748_validate(const unsigned char* bk, const unsigned char* bu, unsigned char* bv) { sim_rfc7748<F_X448, true>(bk, bu, bv); }
void sim_X25519_rfc7748_batch(const unsigned char* bk, const unsigned char* bu, unsigned char* bv, size_t n) {
  for (size_t i = 0; i < n; i++) sim_rfc7748<F_X25519>(bk + 32 * i, bu + 32 * i, bv + 32 * i);
}
void sim_X448_rfc7748_batch(const unsigned char* bk, const unsigned char* bu, unsigned char* bv, size_t n) {
  for (size_t i = 0; i < n; i++) sim_rfc7748<F_X448>(bk + 56 * i, bu + 56 * i, bv + 56 * i);
}
}
