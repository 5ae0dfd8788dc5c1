// Shared device helpers for the demucs_b200 sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define BD_OK 0
#define BD_ERR_ARG -1
#define BD_ERR_CUDA -2

void bd_set_error(const char* fmt, ...);
int bd_check_launch(const char* what);

#define BD_REQUIRE(cond, ...)            \
  do {                                   \
    if (!(cond)) {                       \
      bd_set_error(__VA_ARGS__);         \
      return BD_ERR_ARG;                 \
    }                                    \
  } while (0)

static inline int bd_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// exact-erf GELU, as F.gelu default (reference hdemucs.py:144,334; demucs.py:129; transformer.py:586)
__device__ __forceinline__ float bd_gelu(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
// ex2.approx + rcp.approx: ~2 ulp, a handful of instructions (an IEEE division costs ~40 in a GEMM epilogue)
__device__ __forceinline__ float bd_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float bd_ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// two floats -> packed bf16x2 (round to nearest even), `a` in the low half (the lower address / lower k index)
__device__ __forceinline__ uint32_t bd_pack_bf16(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// round-to-nearest TF32 (low 13 mantissa bits cleared): exactly representable, so the tensor core's own
// fp32 -> tf32 conversion of it is the identity
__device__ __forceinline__ float bd_tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

__device__ __forceinline__ float bd_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double bd_warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of two doubles; result valid in thread 0. `red` = 64 doubles of shared memory.
__device__ __forceinline__ void bd_block_sum2(double& a, double& b, double* red) {
  a = bd_warp_sum_d(a);
  b = bd_warp_sum_d(b);
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) {
    red[warp] = a;
    red[32 + warp] = b;
  }
  __syncthreads();
  if (warp == 0) {
    a = lane < nw ? red[lane] : 0.0;
    b = lane < nw ? red[32 + lane] : 0.0;
    a = bd_warp_sum_d(a);
    b = bd_warp_sum_d(b);
  }
}
