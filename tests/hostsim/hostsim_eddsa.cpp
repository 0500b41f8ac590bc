// tests/hostsim/hostsim_eddsa.cpp -- TEST SCAFFOLDING ONLY (never part of the shipped library).
//
// Eddsa<F_X25519, F_ED25519ORDER>::verify (csrc/eddsa_sm100.cuh) and Edwards::decode (csrc/edwards_sm100.cuh)
// compiled for the host with -DMAB_HOSTSIM, as hostsim.cpp does for the field and group code: the CPU tests
// (tests/test_eddsa.py) run the device-side verification on every fixture row without a GPU.
#define MAB_HOSTSIM 1
#include "gen/field_X25519.cuh"
#include "gen/field_ED25519ORDER.cuh"
#include "eddsa_sm100.cuh"

typedef Eddsa<F_X25519, F_ED25519ORDER> V;
static constexpr int L = V::L;

static void le_words(uint32_t* w, const unsigned char* b, int nw) {
  for (int j = 0; j < nw; j++)
    w[j] = (uint32_t)b[4 * j] | ((uint32_t)b[4 * j + 1] << 8) | ((uint32_t)b[4 * j + 2] << 16) | ((uint32_t)b[4 * j + 3] << 24);
}

static void le_bytes(unsigned char* b, const uint32_t* w, int nw) {
  for (int j = 0; j < 4 * nw; j++) b[j] = (unsigned char)(w[j >> 2] >> (8 * (j & 3)));
}

// h: 64 bytes, sig: 64 bytes R || S, pk: 32 bytes, as RFC 8032 encodes them; table and scratch column in local arrays
extern "C" int sim_ED25519_eddsa_verify(const unsigned char* h, const unsigned char* sig, const unsigned char* pk) {
  uint32_t hw[2 * L], r[L], s[L], a[L];
  le_words(hw, h, 2 * L);
  le_words(r, sig, L);
  le_words(s, sig + 4 * L, L);
  le_words(a, pk, L);
  static uint4 tab[V::M::NE2W * 3 * L / 4];
  static uint32_t scr[V::M::SCR2W];
  return (int)V::verify(hw, r, s, a, tab, 1, scr);
}

// Edwards::decode of a 32-byte encoding: the flag, and the affine point (x, y) as 32 little-endian bytes each
extern "C" int sim_ED25519_decode(const unsigned char* enc, unsigned char* x, unsigned char* y) {
  uint32_t e[L], xw[L], yw[L];
  le_words(e, enc, L);
  V::G::Pt P;
  const uint32_t ok = V::G::decode(P, e);
  V::G::get(xw, yw, P);
  le_bytes(x, xw, L);
  le_bytes(y, yw, L);
  return (int)ok;
}

// k = h mod L of a 64-byte digest, as 32 little-endian bytes
extern "C" void sim_ED25519_reduce512(const unsigned char* h, unsigned char* k) {
  uint32_t hw[2 * L], kw[L];
  le_words(hw, h, 2 * L);
  V::reduce512(kw, hw);
  le_bytes(k, kw, L);
}
