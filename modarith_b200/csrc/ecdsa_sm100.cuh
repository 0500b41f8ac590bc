// ecdsa_sm100.cuh -- batched ECDSA signature verification (SEC1 v2 section 4.1.4; the reference's
// NIST256_VERIFY, nist256.c) over the field FP of the curve and the field FN of its group order, one
// signature per thread.
//
//   ok  = 1 <= r < n  and  1 <= s < n
//   ok &= qx < p  and  qy < p  and  Q on the curve
//   w   = s^-1 mod n,  u1 = h w mod n,  u2 = r w mod n      (h: the digest, leftmost 256 bits; h >= n reduces)
//   R   = u1 G + u2 Q                                       (EcnMul::mul2w, joint 2-bit windows)
//   ok &= Z(R) != 0  and  ( X == r Z  or  (r + n < p and X == (r + n) Z) )
//
// x(R) mod n == r is tested on the homogeneous coordinates: x = X/Z and x < p < 2n, so x mod n == r iff
// x == r or x == r + n -- no inversion of Z, no ecnXXXget.  R = O (Z = 0) must be rejected explicitly: there
// X = 0 = r Z would "match".  Every decision is a mask: the verification runs the same instructions whatever
// the inputs are, like the rest of the library (tools/ct_audit.py treats every loaded value as secret).
#pragma once
#include "mab_field.cuh"
#include "weierstrass_sm100.cuh"

template <class FP, class FN, int PITCH = 0> struct Ecdsa {
  static constexpr int L = FP::L;
  static_assert(L == 8, "P-256: eight 32-bit words");
  static_assert(FN::L == L, "the curve and its group order have the same word count");
  typedef Weierstrass<FP> W;
  typedef Field<FP> Fp;
  typedef Field<FN> Fn;
  typedef EcnMul<W, PITCH> M;
  // resident 128-thread CTAs per SM for k_ecdsa_verify: the setting of k_ecnmul2, which runs the same loop on the
  // same table (168 registers either way); not measured against two CTAs for this kernel
  static constexpr int MINBLOCKS = 3;

  // the P-256 base point as plain little-endian words (FIPS 186-4 D.1.2.3)
  static MAB_DEV void base_point(uint32_t (&gx)[L], uint32_t (&gy)[L]) {
    const uint32_t x[8] = {0xd898c296u, 0xf4a13945u, 0x2deb33a0u, 0x77037d81u, 0x63a440f2u, 0xf8bce6e5u, 0xe12c4247u, 0x6b17d1f2u};
    const uint32_t y[8] = {0x37bf51f5u, 0xcbb64068u, 0x6b315eceu, 0x2bce3357u, 0x7c0f9e16u, 0x8ee7eb4au, 0xfe1a7f9bu, 0x4fe342e2u};
#pragma unroll
    for (int j = 0; j < L; j++) { gx[j] = x[j]; gy[j] = y[j]; }
  }

  // 1 iff (r, s) is a valid signature of digest h under the public key (qx, qy); every argument is a plain value as
  // little-endian words.  tab / pitch / scr / z: the table, scratch column and opaque zero of EcnMul::mul2w.
  static MAB_DEV uint32_t verify(const uint32_t (&h)[L], const uint32_t (&r)[L], const uint32_t (&s)[L],
                                 const uint32_t (&qx)[L], const uint32_t (&qy)[L], uint4* tab, int pitch, uint32_t* scr,
                                 uint32_t z = 0) {
    uint32_t rn[L], sn[L], hn[L], w[L], t[L], u1[L], u2[L];
    uint32_t ok = Fn::from_words(rn, r) & (1u - Fn::is0(rn));
    ok &= Fn::from_words(sn, s) & (1u - Fn::is0(sn));
    (void)Fn::from_words(hn, h);
    Fn::template inv<false>(w, sn, sn);                // s = 0 maps to 0: ok is already 0 there
    FN::mul(t, hn, w);
    Fn::to_words(u1, t);
    FN::mul(t, rn, w);
    Fn::to_words(u2, t);

    typename W::Pt G, Q, R;
    {
      uint32_t gx[L], gy[L];
      base_point(gx, gy);
      W::set(G, gx, gy);
    }
    ok &= W::set_checked(Q, qx, qy);
    M::mul2w(R, u1, G, u2, Q, tab, pitch, scr, z);
    ok &= 1u - Fp::is0_stored(R.z);

    // x(R) == r or x(R) == r + n, as X == r Z or X == (r + n) Z
    uint32_t nw[L], rpn[L], v[L];
    FN::set_p(nw);
    uint32_t carry = 0;
#pragma unroll
    for (int j = 0; j < L; j++) {
      const uint64_t a = (uint64_t)r[j] + nw[j] + carry;
      rpn[j] = (uint32_t)a;
      carry = (uint32_t)(a >> 32);
    }
    (void)Fp::from_words(v, r);                        // r < n < p wherever ok is still 1
    FP::mul(t, v, R.z);
    uint32_t hit = Fp::cmp(t, R.x);
    const uint32_t second = (1u - carry) & Fp::from_words(v, rpn);
    FP::mul(t, v, R.z);
    hit |= second & Fp::cmp(t, R.x);
    return ok & hit;
  }
};

#ifndef MAB_HOSTSIM
#include "mab_kernels.cuh"
// h, r, s, qx, qy: n big-endian 32-byte strings each (the layout of k_ecnmul2); ok[i] = 1 valid, 0 invalid.  Same
// persistent grid and the same 16-entry joint-window table slice per resident CTA in the global workspace as k_ecnmul2;
// shared memory holds the 2L-word scratch column.
template <class FP, class FN> __global__ void __launch_bounds__(MAB_ECN_THREADS, (Ecdsa<FP, FN>::MINBLOCKS))
k_ecdsa_verify(const uint8_t* h, const uint8_t* r, const uint8_t* s, const uint8_t* qx, const uint8_t* qy, uint8_t* ok,
               size_t n, unsigned align, uint4* tabws) {
  constexpr int L = FP::L;
  static_assert(FP::NBYTES == 4 * L, "whole-word byte strings");
  typedef Ecdsa<FP, FN, MAB_ECN_THREADS> V;
  extern __shared__ uint4 mab_smem4[];
  uint4* tab = tabws + (size_t)blockIdx.x * (V::M::NE2W * 3 * (L / 4) * MAB_ECN_THREADS) + threadIdx.x;
  uint32_t* scr = reinterpret_cast<uint32_t*>(mab_smem4) + threadIdx.x;
  for (size_t blk = blockIdx.x; blk * MAB_ECN_THREADS < n; blk += gridDim.x) {
    const size_t i = blk * MAB_ECN_THREADS + threadIdx.x;
    if (i >= n) break;
    uint32_t raw[L], hw[L], rw[L], sw[L], xw[L], yw[L];
    aos_ld<L>(raw, h, i, align);
#pragma unroll
    for (int j = 0; j < L; j++) hw[j] = mab_bswap(raw[L - 1 - j]);
    aos_ld<L>(raw, r, i, align);
#pragma unroll
    for (int j = 0; j < L; j++) rw[j] = mab_bswap(raw[L - 1 - j]);
    aos_ld<L>(raw, s, i, align);
#pragma unroll
    for (int j = 0; j < L; j++) sw[j] = mab_bswap(raw[L - 1 - j]);
    aos_ld<L>(raw, qx, i, align);
#pragma unroll
    for (int j = 0; j < L; j++) xw[j] = mab_bswap(raw[L - 1 - j]);
    aos_ld<L>(raw, qy, i, align);
#pragma unroll
    for (int j = 0; j < L; j++) yw[j] = mab_bswap(raw[L - 1 - j]);
    ok[i] = (uint8_t)V::verify(hw, rw, sw, xw, yw, tab, MAB_ECN_THREADS, scr, align >> 16);   // align <= 16: a zero ptxas cannot fold
  }
}
#endif
