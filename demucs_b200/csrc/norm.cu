// K5: normalisation kernels (HBM-bound; judged on GB/s).
//   GroupNorm(1, C) inside DConv (reference demucs.py:123,138-142), MyGroupNorm(1) norm_out
//   (transformer.py:258-268,372,500), nn.LayerNorm (transformer.py:434-436,591-598) and the
//   LayerScale'd DConv residual update (demucs.py:151-153, transformer.py:236-255).
// Statistics are produced by the producing GEMM's epilogue (sum / sumsq in fp64); here they are
// finalised and applied.
#include "common.cuh"
#include "../../include/demucs_b200.h"

namespace {

__global__ void finalize_group_stats_kernel(double* __restrict__ sums, float* __restrict__ out, int slabs,
                                            double count) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slabs) return;
  double mean = sums[2 * i] / count;
  double var = sums[2 * i + 1] / count - mean * mean;  // biased, as nn.GroupNorm
  if (var < 0.0) var = 0.0;
  out[2 * i] = (float)mean;
  out[2 * i + 1] = (float)(1.0 / sqrt(var + 1e-5));
  sums[2 * i] = 0.0;        // hand the accumulators back cleared: the next producer adds into them directly
  sums[2 * i + 1] = 0.0;
}

// x[m, c] += scale[c] * ( gn(u[m, 2c]) * sigmoid(gn(u[m, 2c+1])) ), gn affine indexed by interleaved column
__global__ void dconv_tail_kernel(float* __restrict__ x, const float* __restrict__ u, const float* __restrict__ mr,
                                  const float* __restrict__ gamma, const float* __restrict__ beta,
                                  const float* __restrict__ scale, long long total2, int C, long long rows_per_item,
                                  int slabs_per_item) {
  // one thread = two output channels (one float4 of u)
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total2) return;
  const int half = C >> 1;
  const long long m = i / half;
  const int c = (int)(i - m * half) * 2;
  // rows are position-major inside an item; its GroupNorm slabs are interleaved with period slabs_per_item
  const long long slab = (m / rows_per_item) * slabs_per_item + (m % slabs_per_item);
  const float mean = __ldg(mr + 2 * slab), rstd = __ldg(mr + 2 * slab + 1);
  const float4 uu = __ldg(reinterpret_cast<const float4*>(u + m * 2 * C + 2 * c));
  const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + 2 * c));
  const float4 bt = __ldg(reinterpret_cast<const float4*>(beta + 2 * c));
  const float2 sc = __ldg(reinterpret_cast<const float2*>(scale + c));
  float a0 = fmaf((uu.x - mean) * rstd, g.x, bt.x), g0 = fmaf((uu.y - mean) * rstd, g.y, bt.y);
  float a1 = fmaf((uu.z - mean) * rstd, g.z, bt.z), g1 = fmaf((uu.w - mean) * rstd, g.w, bt.w);
  float2* xp = reinterpret_cast<float2*>(x + m * C + c);
  float2 xv = *xp;
  xv.x = fmaf(sc.x, a0 * bd_sigmoid(g0), xv.x);
  xv.y = fmaf(sc.y, a1 * bd_sigmoid(g1), xv.y);
  *xp = xv;
}

// h[m, c] = gelu(gn(h[m, c])) in place; one thread = one float4
__global__ void gn_gelu_apply_kernel(float* __restrict__ h, const float* __restrict__ mr,
                                     const float* __restrict__ gamma, const float* __restrict__ beta, long long total4,
                                     int C4, long long rows_per_item, int slabs_per_item) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const long long m = i / C4;
  const int c4 = (int)(i - m * C4);
  const long long slab = (m / rows_per_item) * slabs_per_item + (m % slabs_per_item);
  const float mean = __ldg(mr + 2 * slab), rstd = __ldg(mr + 2 * slab + 1);
  const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c4);
  const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + c4);
  float4* p = reinterpret_cast<float4*>(h) + i;
  float4 v = *p;
  v.x = bd_gelu(fmaf((v.x - mean) * rstd, g.x, b.x));
  v.y = bd_gelu(fmaf((v.y - mean) * rstd, g.y, b.y));
  v.z = bd_gelu(fmaf((v.z - mean) * rstd, g.z, b.z));
  v.w = bd_gelu(fmaf((v.w - mean) * rstd, g.w, b.w));
  *p = v;
}

// One warp per row.  C <= 1024, C % 4 == 0.
template <int MAXV, bool Y16>
__global__ void layer_norm_kernel(const float* __restrict__ x, void* __restrict__ yv, const float* __restrict__ gamma,
                                  const float* __restrict__ beta, const float* __restrict__ pos, int pos_period,
                                  long long M, int C) {
  const long long m = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (m >= M) return;
  const int lane = threadIdx.x & 31;
  const int nv = C >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + m * C);
  float4 v[MAXV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + i * 32;
    if (idx < nv) {
      v[i] = xr[idx];
      s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
  }
  const float mean = bd_warp_sum(s) / C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + i * 32;
    if (idx < nv) {
      float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      q += a * a + b * b + c * c + d * d;
    }
  }
  const float rstd = rsqrtf(bd_warp_sum(q) / C + 1e-5f);
  float4* yr = reinterpret_cast<float4*>(reinterpret_cast<float*>(yv) + (Y16 ? 0 : m * C));
  uint2* yh = reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(yv) + (Y16 ? m * C : 0));
  const float4* pr = pos ? reinterpret_cast<const float4*>(pos + (m % pos_period) * C) : nullptr;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + i * 32;
    if (idx < nv) {
      float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + idx);
      float4 b = __ldg(reinterpret_cast<const float4*>(beta) + idx);
      float4 o;
      o.x = fmaf((v[i].x - mean) * rstd, g.x, b.x);
      o.y = fmaf((v[i].y - mean) * rstd, g.y, b.y);
      o.z = fmaf((v[i].z - mean) * rstd, g.z, b.z);
      o.w = fmaf((v[i].w - mean) * rstd, g.w, b.w);
      if (pr) {
        float4 p = __ldg(pr + idx);
        o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
      }
      if (Y16) {
        yh[idx] = make_uint2(bd_pack_bf16(o.x, o.y), bd_pack_bf16(o.z, o.w));
      } else {
        yr[idx] = o;
      }
    }
  }
}

__global__ void item_stats_kernel(const float* __restrict__ x, double* __restrict__ sums, long long n4) {
  __shared__ double red[64];
  const int b = blockIdx.y;
  const float4* p = reinterpret_cast<const float4*>(x) + (size_t)b * n4;
  double s = 0.0, q = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = __ldg(p + i);
    float ls = v.x + v.y + v.z + v.w;
    float lq = v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    s += ls;
    q += lq;
  }
  bd_block_sum2(s, q, red);
  if (threadIdx.x == 0) {
    atomicAdd(&sums[2 * b], s);
    atomicAdd(&sums[2 * b + 1], q);
  }
}

__global__ void group_norm_apply_kernel(float* __restrict__ x, const float* __restrict__ mr,
                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                        long long per_item4, int C4) {
  const int b = blockIdx.y;
  const float mean = __ldg(mr + 2 * b), rstd = __ldg(mr + 2 * b + 1);
  float4* p = reinterpret_cast<float4*>(x) + (size_t)b * per_item4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_item4;
       i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C4);
    float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c);
    float4 bt = __ldg(reinterpret_cast<const float4*>(beta) + c);
    float4 v = p[i];
    v.x = fmaf((v.x - mean) * rstd, g.x, bt.x);
    v.y = fmaf((v.y - mean) * rstd, g.y, bt.y);
    v.z = fmaf((v.z - mean) * rstd, g.z, bt.z);
    v.w = fmaf((v.w - mean) * rstd, g.w, bt.w);
    p[i] = v;
  }
}

}  // namespace

extern "C" {

int bd_finalize_group_stats(double* sums, float* mean_rstd, int slabs, double count, void* stream) {
  BD_REQUIRE(slabs > 0 && count > 0, "bd_finalize_group_stats: bad sizes");
  finalize_group_stats_kernel<<<bd_cdiv(slabs, 128), 128, 0, (cudaStream_t)stream>>>(sums, mean_rstd, slabs, count);
  return bd_check_launch("finalize_group_stats_kernel");
}

int bd_dconv_tail(float* x, const float* u, const float* mean_rstd, const float* gamma, const float* beta,
                  const float* scale, long long M, int C, long long rows_per_item, int slabs_per_item, void* stream) {
  BD_REQUIRE(C % 4 == 0 && M > 0 && rows_per_item > 0 && slabs_per_item > 0, "bd_dconv_tail: bad sizes (C=%d)", C);
  long long total2 = M * (C / 2);
  dconv_tail_kernel<<<bd_cdiv(total2, 256), 256, 0, (cudaStream_t)stream>>>(x, u, mean_rstd, gamma, beta, scale, total2,
                                                                           C, rows_per_item, slabs_per_item);
  return bd_check_launch("dconv_tail_kernel");
}

int bd_gn_gelu_apply(float* h, const float* mean_rstd, const float* gamma, const float* beta, long long M, int C,
                     long long rows_per_item, int slabs_per_item, void* stream) {
  BD_REQUIRE(C % 4 == 0 && M > 0 && rows_per_item > 0 && slabs_per_item > 0, "bd_gn_gelu_apply: bad sizes (C=%d)", C);
  long long total4 = M * (C / 4);
  gn_gelu_apply_kernel<<<bd_cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(h, mean_rstd, gamma, beta, total4, C / 4,
                                                                              rows_per_item, slabs_per_item);
  return bd_check_launch("gn_gelu_apply_kernel");
}

int bd_layer_norm(const float* x, void* y, const float* gamma, const float* beta, const float* pos, int pos_period,
                  long long M, int C, int y_bf16, void* stream) {
  BD_REQUIRE(C % 4 == 0 && C <= 1024 && M > 0, "bd_layer_norm: C must be a multiple of 4 and <= 1024 (got %d)", C);
  BD_REQUIRE(!pos || pos_period > 0, "bd_layer_norm: pos without period");
  const int warps = 8;
  dim3 grid(bd_cdiv(M, warps));
  const cudaStream_t st = (cudaStream_t)stream;
  if (y_bf16) {
    if (C <= 512) layer_norm_kernel<4, true><<<grid, warps * 32, 0, st>>>(x, y, gamma, beta, pos, pos_period, M, C);
    else layer_norm_kernel<8, true><<<grid, warps * 32, 0, st>>>(x, y, gamma, beta, pos, pos_period, M, C);
  } else {
    if (C <= 512) layer_norm_kernel<4, false><<<grid, warps * 32, 0, st>>>(x, y, gamma, beta, pos, pos_period, M, C);
    else layer_norm_kernel<8, false><<<grid, warps * 32, 0, st>>>(x, y, gamma, beta, pos, pos_period, M, C);
  }
  return bd_check_launch("layer_norm_kernel");
}

int bd_item_stats(const float* x, double* sums, int B, long long n, void* stream) {
  BD_REQUIRE(n % 4 == 0 && B > 0, "bd_item_stats: n must be a multiple of 4");
  int gx = (int)((n / 4 + 256 * 8 - 1) / (256 * 8));
  if (gx > 1184) gx = 1184;  // 8 CTAs per SM x 148
  item_stats_kernel<<<dim3(gx, B), 256, 0, (cudaStream_t)stream>>>(x, sums, n / 4);
  return bd_check_launch("item_stats_kernel");
}

int bd_group_norm_apply(float* x, const float* mean_rstd, const float* gamma, const float* beta, int B,
                        long long rows_per_item, int C, void* stream) {
  BD_REQUIRE(C % 4 == 0 && B > 0, "bd_group_norm_apply: C must be a multiple of 4");
  long long per4 = rows_per_item * (C / 4);
  int gx = (int)((per4 + 256 * 4 - 1) / (256 * 4));
  if (gx > 1184) gx = 1184;
  group_norm_apply_kernel<<<dim3(gx, B), 256, 0, (cudaStream_t)stream>>>(x, mean_rstd, gamma, beta, per4, C / 4);
  return bd_check_launch("group_norm_apply_kernel");
}

}  // extern "C"
