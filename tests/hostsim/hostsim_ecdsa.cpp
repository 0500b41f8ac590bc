// tests/hostsim/hostsim_ecdsa.cpp -- TEST SCAFFOLDING ONLY (never part of the shipped library).
//
// Ecdsa<F_NIST256, F_NIST256ORDER>::verify (csrc/ecdsa_sm100.cuh) compiled for the host with -DMAB_HOSTSIM, as
// hostsim.cpp does for the field and group code: the CPU tests (tests/test_ecdsa.py) run the device-side
// verification on every fixture row without a GPU.
#define MAB_HOSTSIM 1
#include "gen/field_NIST256.cuh"
#include "gen/field_NIST256ORDER.cuh"
#include "ecdsa_sm100.cuh"

// big-endian byte strings in, table and scratch column in local arrays
extern "C" int sim_NIST256_ecdsa_verify(const unsigned char* h, const unsigned char* r, const unsigned char* s,
                                        const unsigned char* qx, const unsigned char* qy) {
  typedef Ecdsa<F_NIST256, F_NIST256ORDER> V;
  constexpr int L = V::L;
  uint32_t w[5][L];
  const unsigned char* src[5] = {h, r, s, qx, qy};
  for (int k = 0; k < 5; k++) {
    for (int j = 0; j < L; j++) w[k][j] = 0;
    for (int b = 0; b < 4 * L; b++) {
      int pos = 4 * L - 1 - b;
      w[k][pos >> 2] |= (uint32_t)src[k][b] << (8 * (pos & 3));
    }
  }
  static uint4 tab[V::M::NE2W * 3 * L / 4];
  static uint32_t scr[V::M::SCR2W];
  return (int)V::verify(w[0], w[1], w[2], w[3], w[4], tab, 1, scr);
}
