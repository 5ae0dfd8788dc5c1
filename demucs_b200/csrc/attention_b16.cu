// K6 (tensor-core arm, bf16 operands): fused attention softmax(Q K^T / 8) V on tcgen05 / TMEM / TMA, head_dim 64.
//
// Same CTA organisation as attention_tc.cu (128 queries of one (item, head) per CTA, key tiles dealt alternately to two
// softmax warpgroups with their own running max / sum and O accumulator in tensor memory, merged at the end), with
// `kind::f16` bf16 operands: K = 16 per instruction at twice the tf32 rate, 128-key tiles, and V consumed as the
// MN-major B operand straight from its natural [key][head_dim] rows (no transpose pass).
//   BD_MATH_BF16X3 (the "strict" mode): a pre-pass splits Q, K and V into bf16 hi = bf16(x) and lo = bf16(x - hi);
//       S = Qlo Khi + Qhi Klo + Qhi Khi, the softmax writes P as a bf16 hi / lo pair (hi over the S columns it came
//       from, lo beside them) and O += Plo Vhi + Phi Vlo + Phi Vhi: 16 mantissa bits per operand, fp32 accumulation.
//   BD_MATH_BF16: single product on the hi parts.
// TMEM (512 columns): X3  [S0|P0hi 128][P0lo 64][S1|P1hi 128][P1lo 64][O0 64][O1 64]
//                     else [S0|P0 128][S1|P1 128][O0 64][O1 64]
// Replaces the SDPA core of nn.MultiheadAttention (reference transformer.py:365,506).
#include <math.h>
#include <stdlib.h>
#include "tcgen05.cuh"
#include "../../include/demucs_b200.h"

namespace {

constexpr int AT_THREADS = 320;                  // warp 0 TMA, warp 1 MMA, warps 2-5 / 6-9 the two softmax groups
constexpr int TQ = 128, HD = 64, TK = 128;
constexpr int TILE = 128 * HD * 2;               // one 128-row x 64-bf16 swizzled box = 16 KB (Q, K and V tiles alike)
constexpr int XCH_LD = 36;                       // floats per row of the final exchange buffer

template <bool X3>
struct BCfg {
  static constexpr int NP = X3 ? 2 : 1;          // operand parts (hi, lo)
  static constexpr int NS = X3 ? 2 : 4;          // K / V stages
  static constexpr int kQBytes = NP * TILE, kKBytes = NP * TILE, kVBytes = NP * TILE;
  static constexpr int kSmem = kQBytes + NS * (kKBytes + kVBytes) + 1024 + 512;
  static_assert(NS * kKBytes >= 2 * TQ * XCH_LD * 4, "exchange buffer reuses the K stages");
};

template <bool X3, bool O16>
__global__ void __launch_bounds__(AT_THREADS, 1) attention_b16_kernel(
    const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_q_lo,
    const __grid_constant__ CUtensorMap map_k_lo, const __grid_constant__ CUtensorMap map_v_lo,
    void* __restrict__ ov, int Tq, int Tk, int ldo) {
  using C_ = BCfg<X3>;
  constexpr int NP = C_::NP, NS = C_::NS;
  constexpr int kQBytes = C_::kQBytes, kKBytes = C_::kKBytes, kVBytes = C_::kVBytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem;                            // [part]
  uint8_t* sK = sQ + kQBytes;                    // [stage][part]
  uint8_t* sV = sK + NS * kKBytes;               // [stage][part]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + NS * kVBytes);
  uint64_t* q_full = bars;                       // [1]
  uint64_t* k_full = bars + 1;                   // [NS]
  uint64_t* v_full = k_full + NS;                // [NS]
  uint64_t* k_empty = v_full + NS;               // [NS]
  uint64_t* v_empty = k_empty + NS;              // [NS]
  uint64_t* s_full = v_empty + NS;               // [2]  one per softmax group
  uint64_t* p_full = s_full + 2;                 // [2]  128 arrivals
  uint64_t* o_final = p_full + 2;                // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_final + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * TQ, h = blockIdx.y, b = blockIdx.z;
  const int ntiles = (Tk + TK - 1) / TK;
  auto col_s = [](int g) { return (uint32_t)(g * (X3 ? 192 : 128)); };          // S / P (hi) of group g
  auto col_plo = [](int g) { return (uint32_t)(g * 192 + 128); };               // X3: P lo
  auto col_o = [](int g) { return (uint32_t)((X3 ? 384 : 256) + g * 64); };

  if (threadIdx.x == 0) {
    for (int i = 0; i < 1 + 4 * NS + 2; ++i) mbar_init(&bars[i], 1);
    mbar_init(&p_full[0], 128);
    mbar_init(&p_full[1], 128);
    mbar_init(&o_final[0], 1);
    mbar_init(&o_final[1], 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    tcgen05_alloc(tmem_slot, 512);
    tcgen05_relinquish();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      mbar_expect_tx(q_full, kQBytes);
#pragma unroll
      for (int p = 0; p < NP; ++p) tma_load_3d(p ? &map_q_lo : &map_q, q_full, sQ + p * TILE, h * HD, q0, b);
      for (int j = 0; j < ntiles; ++j) {
        const int s = j % NS;
        const uint32_t ph = (uint32_t)((j / NS) & 1);
        mbar_wait(&k_empty[s], ph ^ 1);
        mbar_expect_tx(&k_full[s], kKBytes);
#pragma unroll
        for (int p = 0; p < NP; ++p)
          tma_load_3d(p ? &map_k_lo : &map_k, &k_full[s], sK + s * kKBytes + p * TILE, h * HD, j * TK, b);
        mbar_wait(&v_empty[s], ph ^ 1);
        mbar_expect_tx(&v_full[s], kVBytes);
#pragma unroll
        for (int p = 0; p < NP; ++p)
          tma_load_3d(p ? &map_v_lo : &map_v, &v_full[s], sV + s * kVBytes + p * TILE, h * HD, j * TK, b);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc_qk = make_idesc_bf16(TQ, TK);
      constexpr uint32_t idesc_pv = make_idesc_bf16(TQ, HD, 1);      // V: MN-major B operand
      auto issue_qk = [&](int j) {
        const int s = j % NS, g = j & 1;
        mbar_wait(&k_full[s], (uint32_t)((j / NS) & 1));
        tcgen05_fence_after();
        const uint32_t d = tmem + col_s(g);
        const uint8_t* kb = sK + s * kKBytes;
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk) {   // 4 k-steps of 16 head dims = 32 bytes along the swizzled row
          const uint32_t off = 2 * kk;
          const uint64_t a_hi = desc_sw128(sQ) + off;
          const uint64_t b_hi = desc_sw128(kb) + off;
          if (X3) {
            const uint64_t a_lo = desc_sw128(sQ + TILE) + off;
            const uint64_t b_lo = desc_sw128(kb + TILE) + off;
            umma_bf16(d, a_lo, b_hi, idesc_qk, kk != 0);
            umma_bf16(d, a_hi, b_lo, idesc_qk, 1);
            umma_bf16(d, a_hi, b_hi, idesc_qk, 1);
          } else {
            umma_bf16(d, a_hi, b_hi, idesc_qk, kk != 0);
          }
        }
        tcgen05_commit(&s_full[g]);
        tcgen05_commit(&k_empty[s]);
      };
      mbar_wait(q_full, 0);
      issue_qk(0);
      if (ntiles > 1) issue_qk(1);
      for (int j = 0; j < ntiles; ++j) {
        const int s = j % NS, g = j & 1, i = j >> 1;
        mbar_wait(&p_full[g], (uint32_t)(i & 1));
        tcgen05_fence_after();
        mbar_wait(&v_full[s], (uint32_t)((j / NS) & 1));
        tcgen05_fence_after();
        const uint8_t* vb = sV + s * kVBytes;
#pragma unroll
        for (int kk = 0; kk < TK / 16; ++kk) {   // k-steps of 16 keys = 16 rows of V = 2048 bytes; 8 TMEM columns of P
          const uint64_t b_hi = desc_sw128(vb) + (uint32_t)(kk * 128);
          const uint32_t acc = (i | kk) != 0;
          if (X3) {
            const uint64_t b_lo = desc_sw128(vb + TILE) + (uint32_t)(kk * 128);
            umma_bf16_ts(tmem + col_o(g), tmem + col_plo(g) + kk * 8, b_hi, idesc_pv, acc);
            umma_bf16_ts(tmem + col_o(g), tmem + col_s(g) + kk * 8, b_lo, idesc_pv, 1);
            umma_bf16_ts(tmem + col_o(g), tmem + col_s(g) + kk * 8, b_hi, idesc_pv, 1);
          } else {
            umma_bf16_ts(tmem + col_o(g), tmem + col_s(g) + kk * 8, b_hi, idesc_pv, acc);
          }
        }
        tcgen05_commit(&v_empty[s]);
        if (j + 2 >= ntiles) tcgen05_commit(&o_final[g]);
        else issue_qk(j + 2);                    // in order behind P V(j): it overwrites the S/P columns of group g
      }
    }
  } else {
    // ===== softmax warps: two groups of 128 threads, thread = query row =====
    const int g = (warp - 2) >> 2;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const float sl2 = 0.125f * 1.44269504088896340736f;
    const uint32_t s_addr = tmem + lane_addr + col_s(g);
    const uint32_t plo_addr = tmem + lane_addr + col_plo(g);
    const uint32_t o_addr = tmem + lane_addr + col_o(g);
    float m_run = -INFINITY, l_run = 0.f;
    int i = 0;
    for (int j = g; j < ntiles; j += 2, ++i) {
      const int kv_valid = min(TK, Tk - j * TK);
      mbar_wait(&s_full[g], (uint32_t)(i & 1));  // also: every earlier P V of this group has drained
      tcgen05_fence_after();
      // pass 1: row maximum
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
      for (int h0 = 0; h0 < TK; h0 += 64) {
        uint32_t w[64];
        tmem_ld32_nowait(s_addr + h0, w);
        tmem_ld32_nowait(s_addr + h0 + 32, w + 32);
        tmem_ld_wait();
        if (kv_valid < TK) {
#pragma unroll
          for (int c = 0; c < 64; ++c)
            if (h0 + c >= kv_valid) w[c] = 0xff800000u;
        }
#pragma unroll
        for (int c = 0; c < 64; c += 4) {
          mx0 = fmaxf(mx0, __uint_as_float(w[c]));
          mx1 = fmaxf(mx1, __uint_as_float(w[c + 1]));
          mx2 = fmaxf(mx2, __uint_as_float(w[c + 2]));
          mx3 = fmaxf(mx3, __uint_as_float(w[c + 3]));
        }
      }
      const float m_cand = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * sl2;
      const bool raise = m_cand > m_run + 8.0f;   // lazy: P stays below 2^8 with a stale maximum
      if (__any_sync(0xffffffffu, raise)) {
        const float corr = raise ? bd_ex2_approx(m_run - m_cand) : 1.0f;   // first tile: exp2(-inf) = 0
        if (i > 0) {
#pragma unroll
          for (int c0 = 0; c0 < HD; c0 += 32) {
            uint32_t w[32];
            tmem_ld32(o_addr + c0, w);
#pragma unroll
            for (int c = 0; c < 32; ++c) w[c] = __float_as_uint(__uint_as_float(w[c]) * corr);
            tmem_st32(o_addr + c0, w);
          }
        }
        l_run *= corr;
        if (raise) m_run = m_cand;
      }
      // pass 2: P = exp2(S * scale - m), 32 keys at a time with the next chunk's load in flight; the bf16 pairs of
      // chunk c0 land on columns [c0/2, c0/2 + 16) of the S block -- columns this thread has already consumed
      float rs0 = 0.f, rs1 = 0.f, rs2 = 0.f, rs3 = 0.f;
      uint32_t va[32], vb[32];
      tmem_ld32_nowait(s_addr, va);
      tmem_ld_wait();
#pragma unroll
      for (int c0 = 0; c0 < TK; c0 += 32) {
        uint32_t* v = (c0 & 32) ? vb : va;
        uint32_t* vn = (c0 & 32) ? va : vb;
        if (c0 + 32 < TK) tmem_ld32_nowait(s_addr + c0 + 32, vn);
        uint32_t hi[16], lo[X3 ? 16 : 1];
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          const float x0 = fmaf(__uint_as_float(v[c]), sl2, -m_run), x1 = fmaf(__uint_as_float(v[c + 1]), sl2, -m_run);
          const float x2 = fmaf(__uint_as_float(v[c + 2]), sl2, -m_run), x3 = fmaf(__uint_as_float(v[c + 3]), sl2, -m_run);
          float p0 = bd_ex2_approx(x0), p1 = bd_ex2_approx(x1);
          float p2 = bd_ex2_approx(x2), p3 = bd_ex2_approx(x3);
          if (kv_valid < TK) {
            if (c0 + c >= kv_valid) p0 = 0.f;
            if (c0 + c + 1 >= kv_valid) p1 = 0.f;
            if (c0 + c + 2 >= kv_valid) p2 = 0.f;
            if (c0 + c + 3 >= kv_valid) p3 = 0.f;
          }
          rs0 += p0; rs1 += p1; rs2 += p2; rs3 += p3;
          const uint32_t h01 = bd_pack_bf16(p0, p1), h23 = bd_pack_bf16(p2, p3);
          hi[c >> 1] = h01;
          hi[(c >> 1) + 1] = h23;
          if (X3) {
            lo[c >> 1] = bd_pack_bf16(p0 - __uint_as_float(h01 << 16), p1 - __uint_as_float(h01 & 0xffff0000u));
            lo[(c >> 1) + 1] = bd_pack_bf16(p2 - __uint_as_float(h23 << 16), p3 - __uint_as_float(h23 & 0xffff0000u));
          }
        }
        tmem_st16(s_addr + (c0 >> 1), hi);        // P (hi) over consumed S columns
        if (X3) tmem_st16(plo_addr + (c0 >> 1), lo);
        if (c0 + 32 < TK) tmem_ld_wait();
      }
      tmem_st_wait();
      l_run += (rs0 + rs1) + (rs2 + rs3);
      tcgen05_fence_before();
      mbar_arrive(&p_full[g]);
    }
    // ===== merge the two groups' partial results; group g writes head-dim columns [32g, 32g+32) =====
    float own[32], other[32];
    if (i > 0) {
      mbar_wait(&o_final[g], 0);
      tcgen05_fence_after();
      uint32_t w[HD];
      tmem_ld32_nowait(o_addr, w);
      tmem_ld32_nowait(o_addr + 32, w + 32);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        own[c] = __uint_as_float(g ? w[32 + c] : w[c]);
        other[c] = __uint_as_float(g ? w[c] : w[32 + c]);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 32; ++c) own[c] = other[c] = 0.f;
      mbar_wait(&o_final[g ^ 1], 0);             // no tile of our own: still wait until the K stages are idle
    }
    // every Q K^T has completed once any o_final fired (commits cover all earlier MMAs): the K stages are free
    float* xch = reinterpret_cast<float*>(sK);
    float* mine = xch + ((size_t)g * TQ + row) * XCH_LD;
    const float* theirs = xch + ((size_t)(g ^ 1) * TQ + row) * XCH_LD;
#pragma unroll
    for (int c = 0; c < 32; c += 4)               // the half the OTHER group writes out
      *reinterpret_cast<float4*>(mine + c) = make_float4(other[c], other[c + 1], other[c + 2], other[c + 3]);
    mine[32] = m_run;
    mine[33] = l_run;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const float m_o = theirs[32], l_o = theirs[33];
    const float m = fmaxf(m_run, m_o);
    const float w_s = l_run > 0.f ? bd_ex2_approx(m_run - m) : 0.f;
    const float w_o = l_o > 0.f ? bd_ex2_approx(m_o - m) : 0.f;
    const float inv = 1.0f / (l_run * w_s + l_o * w_o);
    const float a_s = w_s * inv, a_o = w_o * inv;
    const int r = q0 + row;
    if (r < Tq) {
      const size_t at = ((size_t)b * Tq + r) * ldo + h * HD + 32 * g;
      if (O16) {
        uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(ov) + at);
#pragma unroll
        for (int c = 0; c < 32; c += 8) {
          const float4 t0 = *reinterpret_cast<const float4*>(theirs + c), t1 = *reinterpret_cast<const float4*>(theirs + c + 4);
          dst[c >> 3] = make_uint4(bd_pack_bf16(fmaf(own[c], a_s, t0.x * a_o), fmaf(own[c + 1], a_s, t0.y * a_o)),
                                   bd_pack_bf16(fmaf(own[c + 2], a_s, t0.z * a_o), fmaf(own[c + 3], a_s, t0.w * a_o)),
                                   bd_pack_bf16(fmaf(own[c + 4], a_s, t1.x * a_o), fmaf(own[c + 5], a_s, t1.y * a_o)),
                                   bd_pack_bf16(fmaf(own[c + 6], a_s, t1.z * a_o), fmaf(own[c + 7], a_s, t1.w * a_o)));
        }
      } else {
        float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(ov) + at);
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          const float4 t = *reinterpret_cast<const float4*>(theirs + c);
          dst[c >> 2] = make_float4(fmaf(own[c], a_s, t.x * a_o), fmaf(own[c + 1], a_s, t.y * a_o),
                                    fmaf(own[c + 2], a_s, t.z * a_o), fmaf(own[c + 3], a_s, t.w * a_o));
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tcgen05_dealloc(tmem, 512);
  }
}

// bf16 [B, T, ld] (columns 0 .. D-1 from `base`) -> boxes of 128 rows x 64 columns, SWIZZLE_128B
bool make_map_b16(CUtensorMap* map, const void* base, int D, int T, int B, int ld = 0) {
  if (!ld) ld = D;
  const cuuint64_t dim[3] = {(cuuint64_t)D, (cuuint64_t)T, (cuuint64_t)B};
  const cuuint64_t str[2] = {(cuuint64_t)ld * 2, (cuuint64_t)T * ld * 2};
  const cuuint32_t box[3] = {64, 128, 1};
  return encode_tensor_map(map, base, 3, dim, str, box, 128, true);
}

// x [rows, ld] (columns 0 .. D-1, fp32) -> dense bf16 hi (and lo = bf16(x - hi)) [rows, D]
template <bool X3>
__global__ void split_rows_b16_kernel(const float* __restrict__ x, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo,
                                      long long rows, int D, int ld) {
  const long long n8 = rows * (D / 8);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / (D / 8);
    const int c = (int)(i - r * (D / 8)) * 8;
    const float4 a = __ldg(reinterpret_cast<const float4*>(x + r * ld + c));
    const float4 e = __ldg(reinterpret_cast<const float4*>(x + r * ld + c + 4));
    const float v[8] = {a.x, a.y, a.z, a.w, e.x, e.y, e.z, e.w};
    uint32_t h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      h[k] = bd_pack_bf16(v[2 * k], v[2 * k + 1]);
      if (X3) l[k] = bd_pack_bf16(v[2 * k] - __uint_as_float(h[k] << 16), v[2 * k + 1] - __uint_as_float(h[k] & 0xffff0000u));
    }
    *reinterpret_cast<uint4*>(hi + r * D + c) = make_uint4(h[0], h[1], h[2], h[3]);
    if (X3) *reinterpret_cast<uint4*>(lo + r * D + c) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

template <bool X3, bool O16>
int launch_attention_b16(const CUtensorMap* m, void* o, int B, int H, int Tq, int Tk, int ldo, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(attention_b16_kernel<X3, O16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       BCfg<X3>::kSmem);
  if (e != cudaSuccess) {
    bd_set_error("bd_attention_b16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return BD_ERR_CUDA;
  }
  dim3 grid((Tq + TQ - 1) / TQ, H, B);
  attention_b16_kernel<X3, O16><<<grid, AT_THREADS, BCfg<X3>::kSmem, st>>>(m[0], m[1], m[2], m[3], m[4], m[5], o, Tq, Tk, ldo);
  return bd_check_launch("attention_b16_kernel");
}

}  // namespace

// Workspace (floats): bf16 copies of Q, K, V (hi, and lo for BD_MATH_BF16X3), D = H*64
long long bd_attention_b16_ws_floats(int B, int H, int Tq, int Tk, int math) {
  const long long D = (long long)H * HD, n = (long long)B * D * (Tq + 2LL * Tk);
  return math == BD_MATH_BF16X3 ? n : (n + 1) / 2;
}

int bd_attention_b16(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk, int ldq,
                     int ldk, int ldv, int ldo, int math, float* ws, void* stream) {
  BD_REQUIRE(B > 0 && H > 0 && Tq > 0 && Tk > 0, "bd_attention: bad sizes");
  BD_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0 && ldo % 4 == 0, "bd_attention: leading dims must be multiples of 4");
  BD_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)o | (uintptr_t)ws) & 15) == 0, "bd_attention: unaligned tensor");
  BD_REQUIRE(ws != nullptr, "bd_attention: the tensor-core arm needs a workspace (see bd_attention_workspace)");
  const cudaStream_t st = (cudaStream_t)stream;
  const bool x3 = math == BD_MATH_BF16X3;
  const int D = H * HD;
  const size_t nq = (size_t)B * Tq * D, nk = (size_t)B * Tk * D;
  uint16_t* base = reinterpret_cast<uint16_t*>(ws);
  uint16_t* q_hi = base;
  uint16_t* k_hi = q_hi + nq;
  uint16_t* v_hi = k_hi + nk;
  uint16_t* q_lo = v_hi + nk;
  uint16_t* k_lo = q_lo + nq;
  uint16_t* v_lo = k_lo + nk;
  if (x3) {
    split_rows_b16_kernel<true><<<148 * 8, 256, 0, st>>>(q, q_hi, q_lo, (long long)B * Tq, D, ldq);
    split_rows_b16_kernel<true><<<148 * 8, 256, 0, st>>>(k, k_hi, k_lo, (long long)B * Tk, D, ldk);
    split_rows_b16_kernel<true><<<148 * 8, 256, 0, st>>>(v, v_hi, v_lo, (long long)B * Tk, D, ldv);
  } else {
    split_rows_b16_kernel<false><<<148 * 8, 256, 0, st>>>(q, q_hi, nullptr, (long long)B * Tq, D, ldq);
    split_rows_b16_kernel<false><<<148 * 8, 256, 0, st>>>(k, k_hi, nullptr, (long long)B * Tk, D, ldk);
    split_rows_b16_kernel<false><<<148 * 8, 256, 0, st>>>(v, v_hi, nullptr, (long long)B * Tk, D, ldv);
  }
  if (bd_check_launch("attention pre-pass") != BD_OK) return BD_ERR_CUDA;
  alignas(64) CUtensorMap m[6];
  bool ok = make_map_b16(&m[0], q_hi, D, Tq, B) && make_map_b16(&m[1], k_hi, D, Tk, B) && make_map_b16(&m[2], v_hi, D, Tk, B);
  if (x3) {
    ok = ok && make_map_b16(&m[3], q_lo, D, Tq, B) && make_map_b16(&m[4], k_lo, D, Tk, B) && make_map_b16(&m[5], v_lo, D, Tk, B);
  } else {
    m[3] = m[0];
    m[4] = m[1];
    m[5] = m[2];
  }
  if (!ok) {
    bd_set_error("bd_attention_b16: TMA tensor map encoding failed");
    return BD_ERR_CUDA;
  }
  return x3 ? launch_attention_b16<true, false>(m, o, B, H, Tq, Tk, ldo, st)
            : launch_attention_b16<false, false>(m, o, B, H, Tq, Tk, ldo, st);
}

// bf16 tensors in, bf16 out: no conversion pass, no workspace
extern "C" int bd_attention_bf16(const void* q, const void* k, const void* v, void* o, int B, int H, int Tq, int Tk, int ldq,
                                 int ldk, int ldv, int ldo, void* stream) {
  BD_REQUIRE(B > 0 && H > 0 && Tq > 0 && Tk > 0, "bd_attention_bf16: bad sizes");
  BD_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 8 == 0, "bd_attention_bf16: leading dims must be multiples of 8");
  BD_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)o) & 15) == 0, "bd_attention_bf16: unaligned tensor");
  const int D = H * HD;
  alignas(64) CUtensorMap m[6];
  if (!(make_map_b16(&m[0], q, D, Tq, B, ldq) && make_map_b16(&m[1], k, D, Tk, B, ldk) && make_map_b16(&m[2], v, D, Tk, B, ldv))) {
    bd_set_error("bd_attention_bf16: TMA tensor map encoding failed");
    return BD_ERR_CUDA;
  }
  m[3] = m[0];
  m[4] = m[1];
  m[5] = m[2];
  return launch_attention_b16<false, true>(m, o, B, H, Tq, Tk, ldo, (cudaStream_t)stream);
}
