// C ABI instantiation for NIST256: generated field code + hand-written kernels.
#include "gen/field_NIST256.cuh"
#include "gen/field_NIST256ORDER.cuh"   // the group order's field, for ECDSA verification
#define MAB_P NIST256
#define MAB_F F_NIST256
#define MAB_HAS_WEIERSTRASS 1
#define MAB_HAS_ECDSA 1
#define MAB_ECDSA_ORDER F_NIST256ORDER

#define MAB_JIT_SRC "jit_src_NIST256.inc"
#include "mab_capi.inc"
