// tests/gpuprobe/blocks.cu -- TEST SCAFFOLDING ONLY (never part of the shipped library).
//
// Runs ONE generated field block (gen/plan.py: mul, sqr, mli, mla, add, sub, neg, canon, add_tt, sub_tt, mul_w,
// sqr_w, and the nres / redc wrappers of gen/emit.py) element-wise on [L, n] limb planes, so that tests can plant
// any stored words -- also the representation edges no public entry point produces -- and compare the words the
// sm_100a build returns with the generator's interpreter (tests/test_gpu_blocks.py).  Compiled once per modulus:
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fPIC -I <gen dir> -I modarith_b200/csrc
//        -DPROBE_HEADER='"field_<NAME>.cuh"' -DPROBE_FIELD=F_<NAME> blocks.cu -o libprobe_<NAME>.so
#include <cuda_runtime.h>
#include PROBE_HEADER

// same order as BLOCKS in tests/test_gpu_blocks.py
enum ProbeOp { P_MUL, P_SQR, P_MLI, P_MLA, P_ADD, P_SUB, P_NEG, P_CANON, P_ADD_TT, P_SUB_TT, P_MUL_W, P_SQR_W, P_NRES,
               P_REDC };

// a, b, c: operand planes (b and c only read by the blocks that take them), s: the small-integer operand of mli / mla
// per element, r: result planes, flag: canon's "input was < p"
template <class F>
__global__ void k_block(int op, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                        const uint32_t* __restrict__ c, const uint32_t* __restrict__ s, uint32_t* __restrict__ r,
                        uint32_t* __restrict__ flag, int n) {
  constexpr int L = F::L;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t x[L], y[L], z[L], o[L];
#pragma unroll
  for (int k = 0; k < L; k++) {
    x[k] = a[(size_t)k * n + i];
    y[k] = b[(size_t)k * n + i];
    z[k] = c[(size_t)k * n + i];
  }
  uint32_t f = 0;
  switch (op) {
    case P_MUL: F::mul(o, x, y); break;
    case P_SQR: F::sqr(o, x); break;
    case P_MLI: F::mli(o, x, s[i]); break;
    case P_MLA: F::mla(o, x, s[i], z); break;
    case P_ADD: F::add(o, x, y); break;
    case P_SUB: F::sub(o, x, y); break;
    case P_NEG: F::neg(o, x); break;
    case P_CANON: f = F::canon(o, x); break;
    case P_ADD_TT: F::add_tt(o, x, y); break;
    case P_SUB_TT: F::sub_tt(o, x, y); break;
    case P_MUL_W: F::mul_w(o, x, y); break;
    case P_SQR_W: F::sqr_w(o, x); break;
    case P_NRES: F::nres(o, x); break;
    case P_REDC: F::redc(o, x); break;
    default: return;
  }
#pragma unroll
  for (int k = 0; k < L; k++) r[(size_t)k * n + i] = o[k];
  flag[i] = f;
}

extern "C" {
int probe_limbs() { return PROBE_FIELD::L; }

// returns the launch's cudaError_t (0 on success)
int probe_block(int op, const void* a, const void* b, const void* c, const void* s, void* r, void* flag, int n,
                void* stream) {
  if (n <= 0) return 0;
  k_block<PROBE_FIELD><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      op, (const uint32_t*)a, (const uint32_t*)b, (const uint32_t*)c, (const uint32_t*)s, (uint32_t*)r,
      (uint32_t*)flag, n);
  return (int)cudaGetLastError();
}
}
