// K6 (exact-fp32 arm): fused softmax(Q K^T / sqrt(64)) V, head_dim 64, no mask, no dropout.
//
// Replaces nn.MultiheadAttention's scaled-dot-product core reached through
// MyTransformerEncoderLayer._sa_block (reference transformer.py:365) and
// CrossTransformerEncoderLayer._ca_block (transformer.py:506); the in/out projections are GEMMs
// (gemm_*.cu).  Flash-style: the [Tq, Tk] score matrix never leaves the SM; the online softmax is
// kept in fp32 in the exp2 domain.  Token counts (2688 / 1344 for htdemucs) are not multiples of
// the tile, the tails are masked.
#include <math.h>
#include "common.cuh"
#include "../../include/demucs_b200.h"

namespace {

constexpr int BQ = 64, BKV = 64, HD = 64, LDS = HD + 4;
constexpr int ATT_THREADS = 256;
constexpr int ATT_SMEM = 4 * BQ * LDS * (int)sizeof(float);

__device__ __forceinline__ void load_tile(float* dst, const float* __restrict__ src, int ld, int rows_valid) {
  // 64 rows x 16 float4, coalesced along the head dimension; rows past the end are zero
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int idx = threadIdx.x + i * ATT_THREADS;
    int row = idx >> 4, c4 = idx & 15;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < rows_valid) v = __ldg(reinterpret_cast<const float4*>(src + (size_t)row * ld) + c4);
    *reinterpret_cast<float4*>(dst + row * LDS + c4 * 4) = v;
  }
}

__global__ void __launch_bounds__(ATT_THREADS) attention_simt_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                                     const float* __restrict__ v, float* __restrict__ o,
                                                                     int Tq, int Tk, int ldq, int ldk, int ldv, int ldo) {
  extern __shared__ __align__(16) float smem[];
  float* sQ = smem;
  float* sK = sQ + BQ * LDS;
  float* sV = sK + BKV * LDS;
  float* sP = sV + BKV * LDS;

  const int q0 = blockIdx.x * BQ, h = blockIdx.y, b = blockIdx.z;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const float* qb = q + ((size_t)b * Tq + q0) * ldq + h * HD;
  const float* kb = k + (size_t)b * Tk * ldk + h * HD;
  const float* vb = v + (size_t)b * Tk * ldv + h * HD;

  load_tile(sQ, qb, ldq, min(BQ, Tq - q0));

  const float sl2 = 0.125f * 1.44269504088896340736f;  // 1/sqrt(64) * log2(e)
  float m_run[4], l_run[4], acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m_run[i] = -INFINITY;
    l_run[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  }

  for (int k0 = 0; k0 < Tk; k0 += BKV) {
    const int kv_valid = min(BKV, Tk - k0);
    __syncthreads();  // previous tile fully consumed (also orders the sQ fill on the first trip)
    load_tile(sK, kb + (size_t)k0 * ldk, ldk, kv_valid);
    load_tile(sV, vb + (size_t)k0 * ldv, ldv, kv_valid);
    __syncthreads();

    // S = Q K^T for rows ty*4+i, columns tx + 16 j
    float s[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 4
    for (int d4 = 0; d4 < HD / 4; ++d4) {
      float4 qa[4], ka[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) qa[i] = *reinterpret_cast<const float4*>(sQ + (ty * 4 + i) * LDS + d4 * 4);
#pragma unroll
      for (int j = 0; j < 4; ++j) ka[j] = *reinterpret_cast<const float4*>(sK + (tx + 16 * j) * LDS + d4 * 4);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          s[i][j] = fmaf(qa[i].x, ka[j].x, s[i][j]);
          s[i][j] = fmaf(qa[i].y, ka[j].y, s[i][j]);
          s[i][j] = fmaf(qa[i].z, ka[j].z, s[i][j]);
          s[i][j] = fmaf(qa[i].w, ka[j].w, s[i][j]);
        }
    }
    // online softmax (exp2 domain)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s[i][j] = (tx + 16 * j < kv_valid) ? s[i][j] * sl2 : -INFINITY;
        mx = fmaxf(mx, s[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float m_new = fmaxf(m_run[i], mx);
      const float corr = exp2f(m_run[i] - m_new);
      float rs = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float p = exp2f(s[i][j] - m_new);
        rs += p;
        sP[(ty * 4 + i) * LDS + tx + 16 * j] = p;
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, off);
      l_run[i] = l_run[i] * corr + rs;
      m_run[i] = m_new;
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] *= corr;
    }
    __syncthreads();
    // O += P V for rows ty*4+i, head columns tx*4 .. tx*4+3
#pragma unroll 4
    for (int c4 = 0; c4 < BKV / 4; ++c4) {
      float4 pa[4], va[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) pa[i] = *reinterpret_cast<const float4*>(sP + (ty * 4 + i) * LDS + c4 * 4);
#pragma unroll
      for (int c = 0; c < 4; ++c) va[c] = *reinterpret_cast<const float4*>(sV + (c4 * 4 + c) * LDS + tx * 4);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(pa[i].x, va[0].x, acc[i][0]); acc[i][1] = fmaf(pa[i].x, va[0].y, acc[i][1]);
        acc[i][2] = fmaf(pa[i].x, va[0].z, acc[i][2]); acc[i][3] = fmaf(pa[i].x, va[0].w, acc[i][3]);
        acc[i][0] = fmaf(pa[i].y, va[1].x, acc[i][0]); acc[i][1] = fmaf(pa[i].y, va[1].y, acc[i][1]);
        acc[i][2] = fmaf(pa[i].y, va[1].z, acc[i][2]); acc[i][3] = fmaf(pa[i].y, va[1].w, acc[i][3]);
        acc[i][0] = fmaf(pa[i].z, va[2].x, acc[i][0]); acc[i][1] = fmaf(pa[i].z, va[2].y, acc[i][1]);
        acc[i][2] = fmaf(pa[i].z, va[2].z, acc[i][2]); acc[i][3] = fmaf(pa[i].z, va[2].w, acc[i][3]);
        acc[i][0] = fmaf(pa[i].w, va[3].x, acc[i][0]); acc[i][1] = fmaf(pa[i].w, va[3].y, acc[i][1]);
        acc[i][2] = fmaf(pa[i].w, va[3].z, acc[i][2]); acc[i][3] = fmaf(pa[i].w, va[3].w, acc[i][3]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = q0 + ty * 4 + i;
    if (r < Tq) {
      const float inv = 1.0f / l_run[i];
      float4 out = make_float4(acc[i][0] * inv, acc[i][1] * inv, acc[i][2] * inv, acc[i][3] * inv);
      *reinterpret_cast<float4*>(o + ((size_t)b * Tq + r) * ldo + h * HD + tx * 4) = out;
    }
  }
}

}  // namespace

int bd_attention_simt(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk, int ldq,
                      int ldk, int ldv, int ldo, void* stream) {
  BD_REQUIRE(B > 0 && H > 0 && Tq > 0 && Tk > 0, "bd_attention: bad sizes");
  BD_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0 && ldo % 4 == 0, "bd_attention: leading dims must be multiples of 4");
  // every row is read and written as float4
  BD_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)o) & 15) == 0, "bd_attention: unaligned tensor");
  cudaError_t e = cudaFuncSetAttribute(attention_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM);
  if (e != cudaSuccess) {
    bd_set_error("bd_attention: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    return BD_ERR_CUDA;
  }
  dim3 grid(bd_cdiv(Tq, BQ), H, B);
  attention_simt_kernel<<<grid, ATT_THREADS, ATT_SMEM, (cudaStream_t)stream>>>(q, k, v, o, Tq, Tk, ldq, ldk, ldv, ldo);
  return bd_check_launch("attention_simt_kernel");
}
