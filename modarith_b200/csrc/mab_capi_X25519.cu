// C ABI instantiation for X25519: generated field code + hand-written kernels.
#include "gen/field_X25519.cuh"
#include "gen/field_ED25519ORDER.cuh"   // the Ed25519 group order's field, for Ed25519 verification (generated
                                        // into the build directory by python -m modarith_b200.build)
#define MAB_P X25519
#define MAB_F F_X25519
#define MAB_HAS_CURVE 1
#define MAB_HAS_EDWARDS 1
#define MAB_HAS_EDDSA 1
#define MAB_EDDSA_ORDER F_ED25519ORDER
#define MAB_JIT_SRC "jit_src_X25519.inc"
#include "mab_capi.inc"
