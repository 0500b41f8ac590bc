// eddsa_sm100.cuh -- batched Ed25519 signature verification (RFC 8032 section 5.1.7, pure Ed25519, the cofactorless
// equation) over the field FP = 2^255 - 19 and the field FN of the group order L, one signature per thread.
//
//   ok  = S < L                                              (S read little-endian; no malleable S + L)
//   ok &= A decodes strictly (Edwards::decode: y < p, x^2 has a root, not x = 0 with the sign bit)
//   k   = h mod L                                            (h = SHA-512(R || A || M) as a 512-bit little-endian value)
//   R'  = [S]B + [k](-A)                                     (EcnMul::mul2w, joint 2-bit windows)
//   ok &= encode(R') == R                                    (all 256 bits: R is never decoded)
//
// Small-order A and R are accepted when the equation holds; no cofactor multiplication is done.  A non-canonical
// or off-curve R never matches, because encode() is canonical.  Every decision is a mask: the verification runs
// the same instructions whatever the inputs are, like the rest of the library (tools/ct_audit.py treats every
// loaded value as secret).
#pragma once
#include "mab_field.cuh"
#include "edwards_sm100.cuh"

template <class FP, class FN, int PITCH = 0> struct Eddsa {
  static constexpr int L = FP::L;
  static_assert(L == 8, "Ed25519: eight 32-bit words");
  static_assert(FN::L == L, "the field and the group order have the same word count");
  typedef Edwards<FP> G;
  typedef Field<FP> Fp;
  typedef Field<FN> Fn;
  typedef EcnMul<G, PITCH> M;

  // the Ed25519 base point as plain little-endian words (RFC 8032 section 5.1)
  static MAB_DEV void base_point(uint32_t (&bx)[L], uint32_t (&by)[L]) {
    const uint32_t x[8] = {0x8f25d51au, 0xc9562d60u, 0x9525a7b2u, 0x692cc760u, 0xfdd6dc5cu, 0xc0a4e231u, 0xcd6e53feu, 0x216936d3u};
#pragma unroll
    for (int j = 0; j < L; j++) { bx[j] = x[j]; by[j] = 0x66666666u; }
    by[0] = 0x66666658u;
  }

  // k = h mod L as plain words: h = h_lo + 2^256 h_hi, and 2^256 h_hi is h_hi (imported, i.e. times R) times R^2
  // under the Montgomery product -- the field's own R^2 constant is the Montgomery form of 2^256
  static MAB_DEV void reduce512(uint32_t (&k)[L], const uint32_t (&h)[2 * L]) {
    uint32_t lo[L], hi[L], r2[L];
#pragma unroll
    for (int j = 0; j < L; j++) { lo[j] = h[j]; hi[j] = h[L + j]; }
    (void)Fn::from_words(lo, lo);
    (void)Fn::from_words(hi, hi);
    FN::set_r2(r2);
    FN::mul(hi, hi, r2);
    FN::add(lo, lo, hi);
    Fn::to_words(k, lo);
  }

  // 1 iff R || S is a valid signature under the encoded public key A for the digest h = SHA-512(R || A || M); every
  // argument is little-endian words as the bytes are given.  tab / pitch / scr / z: the table, scratch column and
  // opaque zero of EcnMul::mul2w.
  static MAB_DEV uint32_t verify(const uint32_t (&h)[2 * L], const uint32_t (&R)[L], const uint32_t (&S)[L],
                                 const uint32_t (&A)[L], uint4* tab, int pitch, uint32_t* scr, uint32_t z = 0) {
    uint32_t k[L], t[L];
    uint32_t ok = Fn::from_words(t, S);             // S < L
    reduce512(k, h);

    typename G::Pt B, NA, Rp;
    ok &= G::decode(NA, A);
    Fp::one(t);
    FP::neg(t, t);
    FP::mul(NA.x, NA.x, t);                          // -A, and a product (tight) again
    {
      uint32_t bx[L], by[L];
      base_point(bx, by);
      (void)Fp::from_words(B.x, bx);
      (void)Fp::from_words(B.y, by);
      Fp::one(B.z);
    }
    M::mul2w(Rp, S, B, k, NA, tab, pitch, scr, z);
    G::encode(t, Rp);
    uint32_t d = 0;
#pragma unroll
    for (int j = 0; j < L; j++) d |= t[j] ^ R[j];
    return ok & (d == 0 ? 1u : 0u);
  }
};

#ifndef MAB_HOSTSIM
#include "mab_kernels.cuh"
// h: n x 64 bytes, sig: n x 64 bytes (R || S), pk: n x 32 bytes, all little-endian as RFC 8032 encodes them;
// ok[i] = 1 valid, 0 invalid.  Same persistent grid, resident CTAs per SM (Edwards::ECN2_MINBLOCKS) and 16-entry
// joint-window table slice per resident CTA in the global workspace as k_ecnmul2<F, Edwards>; shared memory holds
// the 2L-word scratch column.
template <class FP, class FN> __global__ void __launch_bounds__(MAB_ECN_THREADS, Edwards<FP>::ECN2_MINBLOCKS)
k_eddsa_verify(const uint8_t* h, const uint8_t* sig, const uint8_t* pk, uint8_t* ok, size_t n, unsigned align,
               uint4* tabws) {
  constexpr int L = FP::L;
  static_assert(FP::NBYTES == 4 * L, "whole-word byte strings");
  typedef Eddsa<FP, FN, MAB_ECN_THREADS> V;
  extern __shared__ uint4 mab_smem4[];
  uint4* tab = tabws + (size_t)blockIdx.x * (V::M::NE2W * 3 * (L / 4) * MAB_ECN_THREADS) + threadIdx.x;
  uint32_t* scr = reinterpret_cast<uint32_t*>(mab_smem4) + threadIdx.x;
  for (size_t blk = blockIdx.x; blk * MAB_ECN_THREADS < n; blk += gridDim.x) {
    const size_t i = blk * MAB_ECN_THREADS + threadIdx.x;
    if (i >= n) break;
    uint32_t hw[2 * L], sw[2 * L], aw[L], rw[L], s[L];
    aos_ld<2 * L>(hw, h, i, align);
    aos_ld<2 * L>(sw, sig, i, align);
    aos_ld<L>(aw, pk, i, align);
#pragma unroll
    for (int j = 0; j < L; j++) { rw[j] = sw[j]; s[j] = sw[L + j]; }
    ok[i] = (uint8_t)V::verify(hw, rw, s, aw, tab, MAB_ECN_THREADS, scr, align >> 16);   // align <= 16: a zero ptxas cannot fold
  }
}
#endif
