// K6 (tensor-core arm): fused attention softmax(Q K^T / 8) V on tcgen05 / TMEM / TMA, head_dim 64.
//
// One CTA = 128 queries of one (item, head).  The key tiles are dealt alternately to TWO softmax warpgroups
// (split-KV inside the CTA): group g owns tiles j = g, g+2, ... with its own running max / sum and its own
// O accumulator in tensor memory, and the two partial results are merged once at the end.  While group 0 is in
// its softmax the tensor core runs the Q K^T / P V products of group 1 and vice versa, so neither side idles.
//   S = Q K^T      : UMMA 128xTKx8 (tf32), Q and K tiles are K-major SWIZZLE_128B boxes straight from TMA
//   P = softmax    : one query row per thread (TMEM lane = row: row max / sum need no shuffles), exp2 domain,
//                    two passes over the S row in tensor memory (maximum, then exponentials 32 columns at a time
//                    with the next chunk's load in flight); P overwrites S IN PLACE in tensor memory;
//                    the running maximum is only raised when it grows by more than 2^8 (lazy rescale), so the
//                    O accumulator is rarely touched by the softmax warps
//   O += P V       : UMMA 128x64x8 with the A operand read from TMEM (P never touches shared memory) and V^T
//                    tiles as the K-major B operand.  TF32 operands that are MN-major need the special
//                    SWIZZLE_128B_BASE32B layout; instead a small tiled-transpose kernel writes V^T
//                    [B, H*64, Tk] once per call
// BD_MATH_TF32X3 (error-compensated): a pre-pass splits Q, K and V^T into tf32 hi / lo parts; every product
// is issued three times (hi*hi + lo*hi + hi*lo) and the softmax writes P as a hi / lo pair, with 64-key tiles
// so that both parts fit.  TMEM: [S0|P0 .. 128][S1|P1 .. 128][O0 64][O1 64].
// Token counts are not multiples of the tile: TMA zero-fills rows past the item, the softmax masks them.
// Replaces the SDPA core of nn.MultiheadAttention (reference transformer.py:365,506).
#include <math.h>
#include <stdlib.h>
#include "tcgen05.cuh"
#include "../../include/demucs_b200.h"

namespace {

constexpr int AT_THREADS = 320;                  // warp 0 TMA, warp 1 MMA, warps 2-5 / 6-9 the two softmax groups
constexpr int TQ = 128, HD = 64;
constexpr int SUB = TQ * 32 * 4;                 // one 128-row x 32-float swizzled box = 16 KB
constexpr int VSUB = HD * 32 * 4;                // one 64-row x 32-float box of V^T = 8 KB
constexpr int XCH_LD = 36;                       // floats per row of the final exchange buffer

template <bool X3>
struct ACfg {
  static constexpr int TK = X3 ? 64 : 128;       // keys per step
  static constexpr int NP = X3 ? 2 : 1;          // operand parts (hi, lo)
  static constexpr int NS = X3 ? 2 : 3;          // K / V stages
  static constexpr int KSUB = TK * 32 * 4;       // one TK-row x 32-float box of K
  static constexpr int kQBytes = NP * 2 * SUB;
  static constexpr int kKBytes = NP * 2 * KSUB;
  static constexpr int kVBytes = NP * (TK / 32) * VSUB;
  static constexpr int kSmem = kQBytes + NS * (kKBytes + kVBytes) + 1024 + 512;
  static_assert(NS * kKBytes >= 2 * TQ * XCH_LD * 4, "exchange buffer reuses the K stages");
};

template <bool X3>
__global__ void __launch_bounds__(AT_THREADS, 1) attention_tc_kernel(
    const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_q_lo,
    const __grid_constant__ CUtensorMap map_k_lo, const __grid_constant__ CUtensorMap map_v_lo,
    float* __restrict__ o, int Tq, int Tk, int ldo) {
  using C_ = ACfg<X3>;
  constexpr int TK = C_::TK, NP = C_::NP, NS = C_::NS, KSUB = C_::KSUB;
  constexpr int kQBytes = C_::kQBytes, kKBytes = C_::kKBytes, kVBytes = C_::kVBytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem;                            // [part][box]
  uint8_t* sK = sQ + kQBytes;                    // [stage][part][box]
  uint8_t* sV = sK + NS * kKBytes;               // [stage][part][key box]
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
  auto col_s = [](int g) { return (uint32_t)(g * 128); };            // S / P (hi) of group g
  auto col_plo = [](int g) { return (uint32_t)(g * 128 + 64); };     // X3: P lo
  auto col_o = [](int g) { return (uint32_t)(256 + g * 64); };

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
      for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int x = 0; x < 2; ++x)
          tma_load_3d(p ? &map_q_lo : &map_q, q_full, sQ + (p * 2 + x) * SUB, h * HD + 32 * x, q0, b);
      for (int j = 0; j < ntiles; ++j) {
        const int s = j % NS;
        const uint32_t ph = (uint32_t)((j / NS) & 1);
        mbar_wait(&k_empty[s], ph ^ 1);
        mbar_expect_tx(&k_full[s], kKBytes);
#pragma unroll
        for (int p = 0; p < NP; ++p)
#pragma unroll
          for (int x = 0; x < 2; ++x)
            tma_load_3d(p ? &map_k_lo : &map_k, &k_full[s], sK + s * kKBytes + (p * 2 + x) * KSUB, h * HD + 32 * x,
                        j * TK, b);
        mbar_wait(&v_empty[s], ph ^ 1);
        mbar_expect_tx(&v_full[s], kVBytes);
#pragma unroll
        for (int p = 0; p < NP; ++p)
#pragma unroll
          for (int i = 0; i < TK / 32; ++i)      // V^T tile: 64 head-dim rows x TK keys, boxes of 32 keys
            tma_load_3d(p ? &map_v_lo : &map_v, &v_full[s], sV + s * kVBytes + (p * (TK / 32) + i) * VSUB,
                        j * TK + 32 * i, h * HD, b);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc_qk = make_idesc_tf32(TQ, TK);
      constexpr uint32_t idesc_pv = make_idesc_tf32(TQ, HD);
      auto issue_qk = [&](int j) {
        const int s = j % NS, g = j & 1;
        mbar_wait(&k_full[s], (uint32_t)((j / NS) & 1));
        tcgen05_fence_after();
        const uint32_t d = tmem + col_s(g);
        const uint8_t* kb = sK + s * kKBytes;
#pragma unroll
        for (int kk = 0; kk < HD / 8; ++kk) {   // 8 k-steps: two 32-float boxes x 4
          const uint32_t x = kk >> 2, off = 2 * (kk & 3);
          const uint64_t a_hi = desc_sw128(sQ + x * SUB) + off;
          const uint64_t b_hi = desc_sw128(kb + x * KSUB) + off;
          if (X3) {
            const uint64_t a_lo = desc_sw128(sQ + (2 + x) * SUB) + off;
            const uint64_t b_lo = desc_sw128(kb + (2 + x) * KSUB) + off;
            umma_tf32(d, a_lo, b_hi, idesc_qk, kk != 0);
            umma_tf32(d, a_hi, b_lo, idesc_qk, 1);
            umma_tf32(d, a_hi, b_hi, idesc_qk, 1);
          } else {
            umma_tf32(d, a_hi, b_hi, idesc_qk, kk != 0);
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
        for (int kk = 0; kk < TK / 8; ++kk) {   // k-steps of 8 keys
          const uint32_t off = 2 * (kk & 3);
          const uint64_t b_hi = desc_sw128(vb + (kk >> 2) * VSUB) + off;
          const uint32_t acc = (i | kk) != 0;
          if (X3) {
            const uint64_t b_lo = desc_sw128(vb + ((TK / 32) + (kk >> 2)) * VSUB) + off;
            umma_tf32_ts(tmem + col_o(g), tmem + col_plo(g) + kk * 8, b_hi, idesc_pv, acc);
            umma_tf32_ts(tmem + col_o(g), tmem + col_s(g) + kk * 8, b_lo, idesc_pv, 1);
            umma_tf32_ts(tmem + col_o(g), tmem + col_s(g) + kk * 8, b_hi, idesc_pv, 1);
          } else {
            umma_tf32_ts(tmem + col_o(g), tmem + col_s(g) + kk * 8, b_hi, idesc_pv, acc);
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
    const uint32_t o_addr = tmem + lane_addr + col_o(g);
    float m_run = -INFINITY, l_run = 0.f;
    int i = 0;
    for (int j = g; j < ntiles; j += 2, ++i) {
      const int kv_valid = min(TK, Tk - j * TK);
      mbar_wait(&s_full[g], (uint32_t)(i & 1));  // also: every earlier P V of this group has drained
      tcgen05_fence_after();
      // pass 1: row maximum (the S row is read again, chunk by chunk, in pass 2: tensor memory is cheap to read
      // and 128 live values would not leave room for anything else)
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
      // pass 2: P = exp2(S * scale - m) over S in place, 32 columns at a time, the next chunk's load in flight
      float rs0 = 0.f, rs1 = 0.f, rs2 = 0.f, rs3 = 0.f;
      uint32_t va[32], vb[32];
      tmem_ld32_nowait(s_addr, va);
      tmem_ld_wait();
#pragma unroll
      for (int c0 = 0; c0 < TK; c0 += 32) {
        uint32_t* v = (c0 & 32) ? vb : va;
        uint32_t* vn = (c0 & 32) ? va : vb;
        if (c0 + 32 < TK) tmem_ld32_nowait(s_addr + c0 + 32, vn);
        uint32_t lo[X3 ? 32 : 1];
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
          if (X3) {
            const float h0 = bd_tf32_rna(p0), h1 = bd_tf32_rna(p1), h2 = bd_tf32_rna(p2), h3 = bd_tf32_rna(p3);
            v[c] = __float_as_uint(h0); v[c + 1] = __float_as_uint(h1);
            v[c + 2] = __float_as_uint(h2); v[c + 3] = __float_as_uint(h3);
            lo[c] = __float_as_uint(p0 - h0); lo[c + 1] = __float_as_uint(p1 - h1);
            lo[c + 2] = __float_as_uint(p2 - h2); lo[c + 3] = __float_as_uint(p3 - h3);
          } else {
            v[c] = __float_as_uint(p0); v[c + 1] = __float_as_uint(p1);
            v[c + 2] = __float_as_uint(p2); v[c + 3] = __float_as_uint(p3);
          }
        }
        tmem_st32(s_addr + c0, v);               // P (hi) over S, in place
        if (X3) tmem_st32(tmem + lane_addr + col_plo(g) + c0, lo);
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
      float4* dst = reinterpret_cast<float4*>(o + ((size_t)b * Tq + r) * ldo + h * HD + 32 * g);
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        const float4 t = *reinterpret_cast<const float4*>(theirs + c);
        dst[c >> 2] = make_float4(fmaf(own[c], a_s, t.x * a_o), fmaf(own[c + 1], a_s, t.y * a_o),
                                  fmaf(own[c + 2], a_s, t.z * a_o), fmaf(own[c + 3], a_s, t.w * a_o));
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

// fp32 [B, T, ld] (columns 0 .. cols-1 from `base`, items `item_stride` floats apart, default T * ld) -> boxes of
// box_rows rows x 32 columns, SWIZZLE_128B
bool make_map3(CUtensorMap* map, const float* base, int cols, int T, int B, int ld, int box_rows = 128,
               long long item_stride = 0) {
  const cuuint64_t dim[3] = {(cuuint64_t)cols, (cuuint64_t)T, (cuuint64_t)B};
  const cuuint64_t str[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(item_stride ? item_stride : (long long)T * ld) * 4};
  const cuuint32_t box[3] = {32, (cuuint32_t)box_rows, 1};
  return encode_tensor_map(map, base, 3, dim, str, box, 128);
}

// v [B, Tk, ldv] (columns 0 .. D-1) -> vt [B, D, Tkp], 32x32 tiles through shared memory.  SPLIT: write the
// tf32-rounded value to vt and the remainder to vt_lo.
template <bool SPLIT>
__global__ void transpose_v_kernel(const float* __restrict__ v, float* __restrict__ vt, float* __restrict__ vt_lo, int Tk,
                                   int D, int ldv, int Tkp) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8 threads
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + i;
    tile[i][tx] = t < Tk ? __ldg(v + ((size_t)b * Tk + t) * ldv + c0 + tx) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + tx;
    if (t < Tkp) {
      const float x = tile[tx][i];
      const size_t at = ((size_t)b * D + c0 + i) * Tkp + t;
      if (SPLIT) {
        const float hi = bd_tf32_rna(x);
        vt[at] = hi;
        vt_lo[at] = x - hi;
      } else {
        vt[at] = x;
      }
    }
  }
}

// x [B*T rows, ld] (columns 0 .. D-1) -> dense hi / lo [B*T, D] (tf32-rounded value and remainder)
__global__ void split_rows_kernel(const float* __restrict__ x, float* __restrict__ hi, float* __restrict__ lo,
                                  long long rows, int D, int ld) {
  const long long n4 = rows * (D / 4);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / (D / 4);
    const int c = (int)(i - r * (D / 4)) * 4;
    const float4 t = __ldg(reinterpret_cast<const float4*>(x + r * ld + c));
    const float4 h = make_float4(bd_tf32_rna(t.x), bd_tf32_rna(t.y), bd_tf32_rna(t.z), bd_tf32_rna(t.w));
    *reinterpret_cast<float4*>(hi + r * D + c) = h;
    *reinterpret_cast<float4*>(lo + r * D + c) = make_float4(t.x - h.x, t.y - h.y, t.z - h.z, t.w - h.w);
  }
}

template <bool X3>
int launch_attention(const CUtensorMap* m, float* o, int B, int H, int Tq, int Tk, int ldo, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(attention_tc_kernel<X3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       ACfg<X3>::kSmem);
  if (e != cudaSuccess) {
    bd_set_error("bd_attention_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return BD_ERR_CUDA;
  }
  dim3 grid((Tq + TQ - 1) / TQ, H, B);
  attention_tc_kernel<X3><<<grid, AT_THREADS, ACfg<X3>::kSmem, st>>>(m[0], m[1], m[2], m[3], m[4], m[5], o, Tq, Tk, ldo);
  return bd_check_launch("attention_tc_kernel");
}

}  // namespace

// Workspace (floats): BD_MATH_TF32: B*D*Tkp;  BD_MATH_TF32X3: 2*B*D*(Tkp + Tq + Tk), with D = H*64, Tkp = ceil4(Tk).
long long bd_attention_ws_floats(int B, int H, int Tq, int Tk, int math) {
  const long long D = (long long)H * HD, Tkp = (Tk + 3) & ~3;
  return math == BD_MATH_TF32X3 ? 2 * B * D * (Tkp + Tq + Tk) : B * D * Tkp;
}

int bd_attention_tc(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk, int ldq,
                    int ldk, int ldv, int ldo, int math, float* ws, void* stream) {
  BD_REQUIRE(B > 0 && H > 0 && Tq > 0 && Tk > 0, "bd_attention: bad sizes");
  BD_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0 && ldo % 4 == 0, "bd_attention: leading dims must be multiples of 4");
  BD_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)o | (uintptr_t)ws) & 15) == 0, "bd_attention: unaligned tensor");
  BD_REQUIRE(ws != nullptr, "bd_attention: the tensor-core arm needs a workspace (see bd_attention_ws_floats)");
  const cudaStream_t st = (cudaStream_t)stream;
  const bool x3 = math == BD_MATH_TF32X3;
  const int D = H * HD, Tkp = (Tk + 3) & ~3;
  const size_t nvt = (size_t)B * D * Tkp, nq = (size_t)B * Tq * D, nk = (size_t)B * Tk * D;
  float* vt = ws;
  float* vt_lo = ws + nvt;
  float* q_hi = vt_lo + nvt;
  float* q_lo = q_hi + nq;
  float* k_hi = q_lo + nq;
  float* k_lo = k_hi + nk;
  const dim3 tgrid((Tkp + 31) / 32, D / 32, B);
  if (x3) {
    transpose_v_kernel<true><<<tgrid, 256, 0, st>>>(v, vt, vt_lo, Tk, D, ldv, Tkp);
    split_rows_kernel<<<148 * 8, 256, 0, st>>>(q, q_hi, q_lo, (long long)B * Tq, D, ldq);
    split_rows_kernel<<<148 * 8, 256, 0, st>>>(k, k_hi, k_lo, (long long)B * Tk, D, ldk);
  } else {
    transpose_v_kernel<false><<<tgrid, 256, 0, st>>>(v, vt, nullptr, Tk, D, ldv, Tkp);
  }
  if (bd_check_launch("attention pre-pass") != BD_OK) return BD_ERR_CUDA;
  alignas(64) CUtensorMap m[6];
  bool ok;
  if (x3) {
    constexpr int TK = ACfg<true>::TK;
    ok = make_map3(&m[0], q_hi, D, Tq, B, D) && make_map3(&m[1], k_hi, D, Tk, B, D, TK) &&
         make_map3(&m[2], vt, Tk, D, B, Tkp, HD, (long long)D * Tkp) && make_map3(&m[3], q_lo, D, Tq, B, D) &&
         make_map3(&m[4], k_lo, D, Tk, B, D, TK) && make_map3(&m[5], vt_lo, Tk, D, B, Tkp, HD, (long long)D * Tkp);
  } else {
    ok = make_map3(&m[0], q, D, Tq, B, ldq) && make_map3(&m[1], k, D, Tk, B, ldk) &&
         make_map3(&m[2], ws, Tk, D, B, Tkp, HD, (long long)D * Tkp);
    m[3] = m[0];
    m[4] = m[1];
    m[5] = m[2];
  }
  if (!ok) {
    bd_set_error("bd_attention_tc: TMA tensor map encoding failed");
    return BD_ERR_CUDA;
  }
  return x3 ? launch_attention<true>(m, o, B, H, Tq, Tk, ldo, st) : launch_attention<false>(m, o, B, H, Tq, Tk, ldo, st);
}
