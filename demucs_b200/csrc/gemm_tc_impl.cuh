// K3/K4/K7 (tensor-core arm): persistent tcgen05 / TMEM / TMA implicit GEMM for sm_100a, TF32 inputs, fp32
// accumulate.
//
//   out[m, n] = epilogue( sum_k A[m, k] * W[n, k] )      A: activations [M, K] row-major (K-major)
//                                                        W: weights     [N, K] row-major (K-major)
// Both operands are K-major, so one TMA box of 32 (16) floats x 128 rows lands in shared memory as 128-byte
// (64-byte) rows in the SWIZZLE_128B (_64B) pattern that the UMMA shared-memory descriptor consumes directly.
// `tcgen05.mma.cta_group::1.kind::tf32` (M=128, N=TBN, K=8 per instruction) accumulates a 128 x TBN fp32 tile
// in tensor memory.
//
// One CTA per SM walks the tiles (tile = blockIdx.x + i * gridDim.x, column block fastest so that the CTAs
// running at the same time share the activation rows in L2):
//   warp 0      TMA producer (one elected lane); the shared-memory ring (4..16 stages) never drains between tiles
//   warp 1      TMEM allocator + MMA issuer (one elected lane)
//   warps 4..7  (3xTF32) operand splitter: x -> bd_tf32_rna(x), x - hi in shared memory (bf16 modes: warps 2..)
//   last 8..16  epilogue warps, warp w owns TMEM lanes 32*(w%4)..+31.  Wide tiles (TBN >= 64): the 2..4 warps of
//               a lane quarter split the tile's columns and the accumulator is double-buffered, so the epilogue
//               of tile i runs under the main loop of tile i+1.  Tiles of 96 / 192 / 256 columns are finished in
//               chunks of 32 / 64 / 128 so that every warp owns a power-of-two column range.  Narrow tiles
//               (TBN <= 32): each group of 4 warps takes every 4th tile, with 4 accumulators in flight.
// The epilogue dumps its TMEM rows into a staging buffer, then walks them with lane = 4-column group so that
// every global access is a contiguous run of the output row.
//
// Implicit GEMM: for a multi-tap convolution the K loop walks (tap, channel block); the A tile of a tap is ONE
// rank-4 TMA box [channels x R0 positions x R1 rows x 1 item] of the channels-last activation tensor shifted by
// the tap offset (rank 5 with the position split as 4q + r for the stride-4 encoder convolutions) --
// out-of-range coordinates are zero-filled by the TMA unit, which is exactly the convolution's zero padding, so
// there is no im2col buffer and no boundary code.  A 128-row tile is R1 x R0 output positions (R0 = 128 for
// long axes, 8..64 for the short frequency axes of the inner layers).
//
// Covered layers (no A-side transform, C_in % 16 == 0): every nn.Linear of the cross-transformer
// (transformer.py:365,418,506-512), the channel up/down-samplers (htdemucs.py:586-599), the encoder k=8/s=4
// convolutions and 1x1 rewrite + GLU (hdemucs.py:110,152-154), the decoder 3x3 / k=3 rewrite + GLU
// (hdemucs.py:312-313), the transposed convolutions in their 3-tap form (hdemucs.py:326-334), the DConv
// dilated conv3 and, for hidden widths >= 24, its 1x1 expansion (demucs.py:138-153).  C_in <= 8 layers (first
// encoder layer of each branch) stay on the fp32 arm (gemm_simt.cu).
//
// This file is the kernel template + its launcher; it is compiled once per arithmetic family (BD_TC_TU, see
// gemm_tc.cu / gemm_tc_b16x3.cu / gemm_tc_b16.cu) so that the instantiations build in parallel.
//   MODE 0  TF32     kind::tf32, single pass
//   MODE 1  TF32X3   kind::tf32, fp32 hi/lo tiles side by side, 3 products
//   MODE 2  BF16X3   kind::f16 (bf16): the splitter warps turn the fp32 A tile into bf16 hi / lo operands, the
//                    weights arrive pre-split (bf16 hi / lo planes) by TMA; hi*hi + hi*lo + lo*hi.
//                    16 mantissa bits per operand (rel. error ~4e-6 per layer) at 1.5x the cost of one tf32 pass:
//                    the arithmetic of the default ("strict", <= 1e-4) mode.  The three products of a stage read
//                    shared memory heavily, so the main loop is bound by its bandwidth (128 B/clk per SM).  Tiles up
//                    to 192 columns wide (ATM = true) therefore keep the split A operand in TENSOR memory: each
//                    splitter thread converts one row and stores hi | lo with tcgen05.st into a ring of TBK columns
//                    per pipeline stage next to the accumulators, and the MMAs read A from there
//                    (tcgen05.mma [d], [a_tmem], b_desc).  256-column tiles keep the in-place split in shared memory:
//                    their two accumulators already fill the 512 TMEM columns.  ATM = false is the in-place path
//                    at every width (BD_TC_SMEM_A=1 selects it, for comparison).
//   MODE 3  BF16     kind::f16 (bf16), single product (the reduced-precision "bf16" mode)
//   MODE 4  BF16D    the same with a bf16 A tensor in HBM: the tile arrives by TMA in operand form (64 elements =
//                    128-byte rows per k-block), no splitter warps
#pragma once
#include <stdlib.h>
#include "gemm_epilogue.cuh"
#include "tcgen05.cuh"

enum { BD_TC_TF32 = 0, BD_TC_TF32X3 = 1, BD_TC_BF16X3 = 2, BD_TC_BF16 = 3, BD_TC_BF16D = 4 };

struct TileGeom {
  int R0, R1;            // tile = R1 rows (i1) x R0 positions (i0), R0 * R1 == 128, powers of two
  int log2R0;
  int blocks0, blocks1;  // tiles along i0 / i1 per item
  int cpb;               // channel blocks per tap = Cin / TBK
  int stride4;           // 1: k=8/s=4 convolution -- the position axis is viewed as (q, r) = (pos / 4, pos % 4)
};

namespace {

constexpr int TBM = 128;                           // tile rows (UMMA M)

// TBK floats per k-block: 32 -> 128B swizzle, 16 -> 64B swizzle.  TBN = tile columns = UMMA N (16..128):
// narrow outputs (DConv hidden widths, last-layer channels) get narrow tiles instead of zero padding.
// X3: error-compensated "3xTF32": every operand tile is split in shared memory into hi = bd_tf32_rna(x) and
// lo = x - hi and the product is accumulated as hi*hi + lo*hi + hi*lo (fp32-class accuracy, 3x the MMAs).

struct RowInfo {           // per-row epilogue constants, parked in shared memory (32 bytes)
  long long obase;
  int i0;                  // -1: row outside the problem
  int rb_row;
  float e_mean, e_rstd;
  int pad0, pad1;
};

// ---- lean epilogue for the common layer shapes -----------------------------------------------------------
// The generic bd_epi_* helpers test every optional operand per 4-column group; for the layers that dominate the
// run time (plain / GELU / GLU, optional GroupNorm affine, optional LayerScale residual; no transposed-conv
// scatter, channel split, row bias or addend) this version fixes the combination at compile time, keeps
// everything in 32-bit shared-space addresses and predicates instead of branching on row / column validity.
__device__ __forceinline__ float sigmoid_fast(float x) {
  const float e = bd_ex2_approx(-1.44269504088896340736f * x);
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return r;
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}

template <int ACT, bool E, bool RES, bool ROWB, bool CT, int WC, int RB>
__device__ __forceinline__ void epi_fast_rows(const bd_gemm_desc& d, uint32_t stage_s, uint32_t rinfo_s, int lane, int n0w,
                                              float& ssum, float& ssq) {
  constexpr int LDT = WC + 4;
  constexpr int CG = WC / 4 < 32 ? WC / 4 : 32;   // lanes across the warp's columns
  constexpr int RPI = 32 / CG;                    // rows per pass
  const int cg = lane % CG, rsub = lane / CG;
  const int n = n0w + 4 * cg;
  const bool col_ok = n < d.N;
  const int nc = col_ok ? n : 0;                  // clamped: operands are fetched unconditionally
  const float4 bias = d.bias ? ldg4(d.bias + nc) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 gam = make_float4(1.f, 1.f, 1.f, 1.f), bet = make_float4(0.f, 0.f, 0.f, 0.f);
  if (E) {
    gam = ldg4(d.e_gamma + nc);
    bet = ldg4(d.e_beta + nc);
  }
  const int no = ACT == BD_ACT_GLU ? nc >> 1 : nc;
  float4 scl = make_float4(1.f, 1.f, 1.f, 1.f);
  if (RES && d.scale) {
    if (ACT == BD_ACT_GLU) {
      const float2 t = ldg2(d.scale + no);
      scl.x = t.x; scl.y = t.y;
    } else {
      scl = ldg4(d.scale + no);
    }
  }
  // transposed conv: column n = (output phase rr, channel); the row offset already points at phase 0
  int rr = 0;
  long long colofs = no;
  if (CT) {
    const int cout = d.N >> 2;
    rr = nc / cout;
    colofs = (long long)rr * d.os_0 + (nc - rr * cout);
    rr -= d.convt == 1 ? 2 : 0;
  }
  const long long outo = colofs;
  const float* resp = RES ? d.resid + colofs : nullptr;
  const float* addp = CT && d.addend ? d.addend + colofs : nullptr;
  const float* rbp = ROWB ? d.rowbias + no : nullptr;
  const int rb_ld = ACT == BD_ACT_GLU ? d.N >> 1 : d.N;
  const uint32_t st_lane = stage_s + (uint32_t)(rsub * LDT + 4 * cg) * 4u;
  const uint32_t ri_lane = rinfo_s + (uint32_t)rsub * 32u;
#pragma unroll 1
  for (int it = 0; it < 32 / RPI; it += RB) {
    long long ob[RB];
    bool ok[RB];
    float mean[RB], rstd[RB];
    float4 res[RB];   // residual / row bias / skip operand (at most one of them per combination)
#pragma unroll
    for (int u = 0; u < RB; ++u) {
      const uint32_t ra = ri_lane + (uint32_t)((it + u) * RPI) * 32u;
      uint32_t w0, w1, w2, w3;
      asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "r"(ra));
      ob[u] = (long long)(((unsigned long long)w1 << 32) | w0);
      ok[u] = (int)w2 >= 0 && col_ok;
      if (CT) ok[u] = ok[u] && (unsigned)(4 * (int)w2 + rr) < (unsigned)d.O0;
      if (ROWB || CT) res[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ROWB && ok[u]) {
        if (ACT == BD_ACT_GLU) {
          const float2 t = ldg2(rbp + (size_t)w3 * rb_ld);
          res[u].x = t.x; res[u].y = t.y;
        } else {
          res[u] = ldg4(rbp + (size_t)w3 * rb_ld);
        }
      }
      if (CT && addp && ok[u]) res[u] = ldg4(addp + ob[u]);
      if (E) asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(mean[u]), "=f"(rstd[u]) : "r"(ra + 16));
      if (RES) {
        res[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok[u]) {
          if (ACT == BD_ACT_GLU) {
            const float2 t = ldg2(resp + ob[u]);
            res[u].x = t.x; res[u].y = t.y;
          } else {
            res[u] = ldg4(resp + ob[u]);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < RB; ++u) {
      float4 v = lds128(st_lane + (uint32_t)((it + u) * RPI * LDT) * 4u);
      v.x += bias.x; v.y += bias.y; v.z += bias.z; v.w += bias.w;
      if (E) {
        v.x = fmaf((v.x - mean[u]) * rstd[u], gam.x, bet.x);
        v.y = fmaf((v.y - mean[u]) * rstd[u], gam.y, bet.y);
        v.z = fmaf((v.z - mean[u]) * rstd[u], gam.z, bet.z);
        v.w = fmaf((v.w - mean[u]) * rstd[u], gam.w, bet.w);
      }
      if (ACT == BD_ACT_GLU) {
        float2 o2 = make_float2(v.x * sigmoid_fast(v.y), v.z * sigmoid_fast(v.w));
        if (ROWB) {
          o2.x += res[u].x;
          o2.y += res[u].y;
        }
        if (RES) {
          o2.x = fmaf(scl.x, o2.x, res[u].x);
          o2.y = fmaf(scl.y, o2.y, res[u].y);
        }
        if (ok[u]) {
          bd_store_out2(d, outo + ob[u], o2);
          ssum += o2.x + o2.y;
          ssq = fmaf(o2.x, o2.x, fmaf(o2.y, o2.y, ssq));
        }
      } else {
        if (ACT == BD_ACT_GELU) {
          v.x = bd_gelu(v.x); v.y = bd_gelu(v.y); v.z = bd_gelu(v.z); v.w = bd_gelu(v.w);
        }
        if (RES) {
          v.x = fmaf(scl.x, v.x, res[u].x); v.y = fmaf(scl.y, v.y, res[u].y);
          v.z = fmaf(scl.z, v.z, res[u].z); v.w = fmaf(scl.w, v.w, res[u].w);
        }
        if (ROWB || CT) {
          v.x += res[u].x; v.y += res[u].y; v.z += res[u].z; v.w += res[u].w;
        }
        if (ok[u]) {
          bd_store_out4(d, outo + ob[u], v);
          ssum += (v.x + v.y) + (v.z + v.w);
          ssq = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, ssq))));
        }
      }
    }
  }
}

// which compile-time combination (if any) covers this launch; uniform per kernel
__device__ __forceinline__ int epi_fast_id(const bd_gemm_desc& d, bool vec, bool row_stats) {
  if (!vec || row_stats || !d.out || d.oc_split) return -1;
  const bool e = d.e_stats != nullptr, r = d.resid != nullptr;
  if (d.convt) return (d.act == BD_ACT_GELU && !e && !r && !d.rowbias) ? 6 : -1;
  if (d.addend) return -1;
  if (d.rowbias) return (d.act == BD_ACT_GLU && !e && !r) ? 5 : -1;
  if (d.act == BD_ACT_NONE && !e) return r ? 1 : 0;
  if (d.act == BD_ACT_GELU && !e && !r) return 2;
  if (d.act == BD_ACT_GLU && !e && !r) return 3;
  if (d.act == BD_ACT_GLU && e && r) return 4;
  return -1;
}

// ---- persistent variant ----------------------------------------------------------------------------------
// One CTA per SM walks tiles tile = blockIdx.x, blockIdx.x + gridDim.x, ...  The shared-memory ring never
// drains between tiles, the accumulator is double-buffered in TMEM (2 x TBN columns), and the epilogue of tile i
// (warps 4..7, dedicated staging buffer) runs while the MMA warp is already accumulating tile i+1.
#ifndef BD_TC_EPI_GROUPS
#define BD_TC_EPI_GROUPS 4
#endif
// Epilogue warps per TMEM lane quarter (column split): 4 in the single-pass kernel, where the epilogue is the
// bottleneck; the 3xTF32 kernel spends 3x longer per tile on the tensor core, so 2 suffice and 4 more warps
// split the fp32 operand tiles into tf32 hi / lo parts in shared memory.
__host__ __device__ constexpr int pow2_at_least(int v, int p) { return p >= v ? p : pow2_at_least(v, 2 * p); }

template <int TBK, int TBN, int MODE, bool ATM = false>
struct PCfg {
  static_assert(!ATM || (MODE == BD_TC_BF16X3 && TBN <= 192), "A in tensor memory: strict mode, tiles up to 192 wide");
  static_assert(TBN % 16 == 0 && TBN <= 256, "UMMA N (M = 128): a multiple of 16 up to 256");
  static constexpr bool kX3 = MODE == BD_TC_TF32X3;                          // fp32 hi / lo tiles side by side
  static constexpr bool kB16 = MODE == BD_TC_BF16X3 || MODE == BD_TC_BF16 || MODE == BD_TC_BF16D;   // bf16 operands
  static constexpr bool kDirect = MODE == BD_TC_BF16D;                       // A is bf16 in HBM
  static constexpr bool kSplit = MODE != BD_TC_TF32 && !kDirect;             // splitter warps present
  static constexpr int kBParts = MODE == BD_TC_BF16X3 ? 2 : 1;               // bf16 weight planes per stage (hi, lo)
  static constexpr int kPGroups = (MODE == BD_TC_TF32X3 || MODE == BD_TC_BF16X3) ? 2 : BD_TC_EPI_GROUPS;
  // warps: 0 TMA, 1 MMA, then the splitters (3xTF32: warps 4..7; bf16x3: warps 2..5; bf16: warps 2..3 -- one
  // product per stage leaves them half the conversion work and the epilogue needs the registers), then the epilogue
  static constexpr int kSplitWarp0 = kB16 ? 2 : 4;
  static constexpr int kSplitWarps = MODE == BD_TC_BF16 ? 2 : 4;
  static constexpr int kEpiWarp0 = kSplit ? kSplitWarp0 + kSplitWarps : 4;
  static constexpr int kThreads = 32 * kEpiWarp0 + 128 * kPGroups;
  static constexpr int kTileBytesA = TBM * TBK * (kDirect ? 2 : 4);          // fp32 from TMA (bf16 modes: split in place)
  static constexpr int kTileBytesB = kB16 ? TBN * TBK * 2 : TBN * TBK * 4;
  static constexpr int kStageBytesA = (kX3 ? 2 : 1) * kTileBytesA;
  static constexpr int kStageBytesB = (kX3 ? 2 : kBParts) * kTileBytesB;
  static constexpr int kTxBytes = kTileBytesA + (kB16 ? kBParts : 1) * kTileBytesB;   // TMA bytes per stage
  // wide tiles: the epilogue groups split the COLUMNS of one tile (two accumulators, ping-pong); narrow tiles
  // (TBN <= 32, the epilogue of one tile is too small to share): each group takes every kPGroups-th TILE
  static constexpr bool kTileSplit = TBN <= 32;
  static constexpr int kNAcc = kTileSplit ? kPGroups : 2;
  // columns the epilogue finishes at a time: every warp of a lane quarter must own a power of two >= 16 of them
  static constexpr int kChunk = TBN == 256 ? 128 : TBN == 192 ? 64 : TBN == 96 ? 32 : TBN;
  static constexpr int kChunks = TBN / kChunk;
  static constexpr int kWarpCols = kTileSplit ? TBN : kChunk / kPGroups;
  static_assert(kWarpCols >= 16 && (kWarpCols & (kWarpCols - 1)) == 0, "epilogue: power-of-two warp column range");
  static constexpr int kStagingBytes = 4 * kPGroups * 32 * (kWarpCols + 4) * 4;
  static constexpr int kTailBytes = 512 + 128 * kPGroups * 32;   // barriers + TMEM slot, then the row tables
  static constexpr int kBudget = 227 * 1024 - 1024 - kTailBytes - kStagingBytes;
  static constexpr int kStagesRaw = kBudget / (kStageBytesA + kStageBytesB);
  static constexpr int kStages = kStagesRaw > (kTileSplit ? 16 : 8) ? (kTileSplit ? 16 : 8) : kStagesRaw;
  static constexpr int kSmemBytes = kStages * (kStageBytesA + kStageBytesB) + kStagingBytes + 1024 + kTailBytes;
  // ATM: the A ring in tensor memory has one slot per shared-memory stage (TBK columns = TBK/2 hi + TBK/2 lo, two
  // bf16 per column) after the accumulators, so the stage's empty barrier also frees its A slot
  static constexpr int kACol0 = kNAcc * TBN;
  static constexpr int kTmemUsed = kNAcc * TBN + (ATM ? kStages * TBK : 0);
  static_assert(kTmemUsed <= 512, "tensor memory: accumulators + A ring exceed 512 columns");
  static constexpr int kTmemCols = pow2_at_least(kTmemUsed, 32);   // the allocation is a power of two >= 32
};

template <int TBK, int TBN, int MODE, bool ATM>
__global__ void __launch_bounds__((PCfg<TBK, TBN, MODE, ATM>::kThreads), 1) conv_gemm_tc_persist_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                            const __grid_constant__ CUtensorMap map_b,
                                                                            const __grid_constant__ CUtensorMap map_b_lo,
                                                                            const bd_gemm_desc d, const TileGeom g,
                                                                            int ntiles, int ntn) {
  using C_ = PCfg<TBK, TBN, MODE, ATM>;
  constexpr bool X3 = C_::kX3, B16 = C_::kB16, SPLIT = C_::kSplit;
  constexpr int kPGroups = C_::kPGroups;
  constexpr int kTileBytesA = C_::kTileBytesA, kTileBytesB = C_::kTileBytesB;
  constexpr int kStages = C_::kStages, kStageBytesA = C_::kStageBytesA, kStageBytesB = C_::kStageBytesB;
  constexpr int kTmemCols = C_::kTmemCols;
  constexpr int WC = C_::kWarpCols;               // columns one epilogue warp owns
  constexpr int CW = WC < 32 ? WC : 32;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + kStages * kStageBytesA;
  float* staging = reinterpret_cast<float*>(sB + kStages * kStageBytesB);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(staging) + C_::kStagingBytes);
  uint64_t* empty_bar = full_bar + kStages;
  constexpr int kNAcc = C_::kNAcc;
  constexpr bool kTileSplit = C_::kTileSplit;
  constexpr int NCH = C_::kChunks, CHW = C_::kChunk;
  uint64_t* tmem_full = empty_bar + kStages;       // [kNAcc]
  uint64_t* tmem_empty = tmem_full + kNAcc;        // [kNAcc]
  uint64_t* conv_bar = tmem_empty + kNAcc;             // [kStages] X3: hi/lo tiles written by the splitter warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(conv_bar + kStages);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = d.taps * g.cpb;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
      mbar_init(&conv_bar[s], 32 * C_::kSplitWarps);
    }
    for (int a = 0; a < kNAcc; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], kTileSplit ? 4 : 4 * kPGroups);   // one arrival per epilogue warp of the tile
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tcgen05_alloc(tmem_slot, kTmemCols);
    tcgen05_relinquish();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // tile -> (column block fastest, then position block, row block, item)
  auto decode = [&](int tile, int& b, int& i0s, int& i1s, int& n0) {
    const int nb = tile % ntn;
    int r = tile / ntn;
    const int blk0 = r % g.blocks0;
    r /= g.blocks0;
    const int blk1 = r % g.blocks1;
    b = r / g.blocks1;
    i0s = blk0 * g.R0;
    i1s = blk1 * g.R1;
    n0 = nb * TBN;
  };

  if (warp == 0) {
    // ===== TMA producer: the ring runs straight through tile boundaries =====
    if (lane == 0) {
      long long kbg = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        int b, i0s, i1s, n0;
        decode(tile, b, i0s, i1s, n0);
        int tap = 0, cb = 0;
        for (int kb = 0; kb < nkb; ++kb, ++kbg) {
          const int s = (int)(kbg % kStages);
          const uint32_t ph = (uint32_t)((kbg / kStages) & 1);
          mbar_wait_parked(&empty_bar[s], ph ^ 1);
          mbar_expect_tx(&full_bar[s], C_::kTxBytes);
          if (g.stride4) {
            const int d0 = d.d0[tap];
            tma_load_5d(&map_a, &full_bar[s], sA + s * kStageBytesA, cb * TBK, d0 & 3, i0s + (d0 >> 2), i1s + d.d1[tap], b);
          } else {
            tma_load_4d(&map_a, &full_bar[s], sA + s * kStageBytesA, cb * TBK, i0s + d.d0[tap], i1s + d.d1[tap], b);
          }
          tma_load_2d(&map_b, &full_bar[s], sB + s * kStageBytesB, tap * d.Cin + cb * TBK, n0);
          if constexpr (MODE == BD_TC_BF16X3)
            tma_load_2d(&map_b_lo, &full_bar[s], sB + s * kStageBytesB + kTileBytesB, tap * d.Cin + cb * TBK, n0);
          if (++cb == g.cpb) {
            cb = 0;
            ++tap;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc = B16 ? make_idesc_bf16(TBM, TBN) : make_idesc_tf32(TBM, TBN);
      long long kbg = 0;
      int tcount = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
        const int a = tcount % kNAcc;
        mbar_wait_parked(&tmem_empty[a], (uint32_t)(((tcount / kNAcc) & 1) ^ 1));   // epilogue has drained this accumulator
        tcgen05_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(a * TBN);
        for (int kb = 0; kb < nkb; ++kb, ++kbg) {
          const int s = (int)(kbg % kStages);
          const uint32_t ph = (uint32_t)((kbg / kStages) & 1);
          mbar_wait_parked(SPLIT ? &conv_bar[s] : &full_bar[s], ph);
          tcgen05_fence_after();
          if constexpr (ATM) {
            // A: TMEM slot s = [hi: TBK/2 columns | lo: TBK/2 columns]; B: dense bf16 planes
            const uint32_t a_hi = tmem_base + (uint32_t)(C_::kACol0 + s * TBK), a_lo = a_hi + TBK / 2;
            const uint64_t b_hi = make_kmajor_desc16<TBK>(sB + s * kStageBytesB, 8 * TBK * 2);
            const uint64_t b_lo = make_kmajor_desc16<TBK>(sB + s * kStageBytesB + kTileBytesB, 8 * TBK * 2);
#pragma unroll
            for (int k = 0; k < TBK / 16; ++k) {
              umma_bf16_ts(acc, a_lo + 8 * k, b_hi + 2 * k, idesc, (kb | k) != 0);   // small terms first
              umma_bf16_ts(acc, a_hi + 8 * k, b_lo + 2 * k, idesc, 1);
              umma_bf16_ts(acc, a_hi + 8 * k, b_hi + 2 * k, idesc, 1);
            }
          } else if constexpr (B16) {
            // A: 8-row groups of [hi 8 x TBK bf16 | lo 8 x TBK bf16] where the fp32 rows were; B: dense bf16 planes
            const uint64_t a_hi = make_kmajor_desc16<TBK>(sA + s * kStageBytesA, C_::kDirect ? 8 * TBK * 2 : 8 * TBK * 4);
            const uint64_t a_lo = make_kmajor_desc16<TBK>(sA + s * kStageBytesA + 8 * TBK * 2, 8 * TBK * 4);
            const uint64_t b_hi = make_kmajor_desc16<TBK>(sB + s * kStageBytesB, 8 * TBK * 2);
            const uint64_t b_lo = make_kmajor_desc16<TBK>(sB + s * kStageBytesB + kTileBytesB, 8 * TBK * 2);
#pragma unroll
            for (int k = 0; k < TBK / 16; ++k) {
              if constexpr (MODE == BD_TC_BF16X3) {
                umma_bf16(acc, a_lo + 2 * k, b_hi + 2 * k, idesc, (kb | k) != 0);   // small terms first
                umma_bf16(acc, a_hi + 2 * k, b_lo + 2 * k, idesc, 1);
                umma_bf16(acc, a_hi + 2 * k, b_hi + 2 * k, idesc, 1);
              } else {
                umma_bf16(acc, a_hi + 2 * k, b_hi + 2 * k, idesc, (kb | k) != 0);
              }
            }
          } else {
          const uint64_t adesc = make_kmajor_desc<TBK>(sA + s * kStageBytesA);
          const uint64_t bdesc = make_kmajor_desc<TBK>(sB + s * kStageBytesB);
#pragma unroll
          for (int k = 0; k < TBK / 8; ++k) {
            if constexpr (X3) {
              const uint64_t alo = make_kmajor_desc<TBK>(sA + s * kStageBytesA + kTileBytesA);
              const uint64_t blo = make_kmajor_desc<TBK>(sB + s * kStageBytesB + kTileBytesB);
              umma_tf32(acc, alo + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);   // small terms first
              umma_tf32(acc, adesc + 2 * k, blo + 2 * k, idesc, 1);
              umma_tf32(acc, adesc + 2 * k, bdesc + 2 * k, idesc, 1);
            } else {
              umma_tf32(acc, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
            }
          }
          }
          tcgen05_commit(&empty_bar[s]);
        }
        tcgen05_commit(&tmem_full[a]);
      }
    }
  } else if (SPLIT && warp >= C_::kSplitWarp0 && warp < C_::kSplitWarp0 + C_::kSplitWarps) {
    const int et = threadIdx.x - 32 * C_::kSplitWarp0;      // 0..127
    long long kbg = 0;
    if constexpr (ATM) {
      // ===== operand splitter, A in tensor memory: one thread per tile row =====
      // Warp w may only touch TMEM lanes 32*(w%4)..+31, so it converts those rows: the thread reads its row's TBK
      // floats (16-byte chunks in the TMA swizzle: 8 consecutive rows hit 8 different chunk positions, no bank
      // conflict) and stores bf16 hi | lo into the stage's TMEM slot.  The slot is free once full_bar[s] completes:
      // the producer refilled stage s only after the MMAs that last read the slot committed empty_bar[s].
      static_assert(TBK == 16 || TBK == 32, "A in tensor memory: 16 or 32 columns per stage");
      constexpr int RB = TBK * 4;                          // bytes per fp32 row
      const int row = 32 * (warp & 3) + lane;
      const int xr = (row * RB >> 7) & (RB / 16 - 1);      // swizzle XOR term of the row
      const uint32_t lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
      (void)et;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int kb = 0; kb < nkb; ++kb, ++kbg) {
          const int s = (int)(kbg % kStages);
          mbar_wait(&full_bar[s], (uint32_t)((kbg / kStages) & 1));
          const uint8_t* rp = sA + s * kStageBytesA + row * RB;
          uint32_t hl[TBK];                                // [hi: TBK/2 columns | lo: TBK/2 columns]
#pragma unroll
          for (int j = 0; j < TBK / 4; ++j) {
            const float4 x = *reinterpret_cast<const float4*>(rp + ((j ^ xr) << 4));
            const uint32_t h0 = bd_pack_bf16(x.x, x.y), h1 = bd_pack_bf16(x.z, x.w);
            hl[2 * j] = h0;
            hl[2 * j + 1] = h1;
            hl[TBK / 2 + 2 * j] = bd_pack_bf16(x.x - __uint_as_float(h0 << 16), x.y - __uint_as_float(h0 & 0xffff0000u));
            hl[TBK / 2 + 2 * j + 1] = bd_pack_bf16(x.z - __uint_as_float(h1 << 16), x.w - __uint_as_float(h1 & 0xffff0000u));
          }
          tcgen05_fence_after();
          const uint32_t slot = tmem_base + lane_addr + (uint32_t)(C_::kACol0 + s * TBK);
          if constexpr (TBK == 32) tmem_st32(slot, hl); else tmem_st16(slot, hl);
          tmem_st_wait();
          tcgen05_fence_before();
          mbar_arrive(&conv_bar[s]);
        }
      }
    } else if constexpr (B16) {
      // ===== operand splitter (bf16 modes): the fp32 A tile becomes bf16 hi (and lo = bf16(x - hi)) IN PLACE =====
      // An 8-row group of the fp32 tile (8 * TBK * 4 bytes, TMA-swizzled) is rewritten as [8 x TBK bf16 hi | 8 x TBK
      // bf16 lo], each half in the K-major swizzle of its own row size.  One warp owns a whole group, so loading the
      // group into registers, __syncwarp, then storing is all the ordering the in-place rewrite needs.
      constexpr int RB = TBK * 4, RH = TBK * 2;            // bytes per fp32 row / per bf16 row
      constexpr int GB = 8 * RB;                           // bytes per group
      constexpr int SW = C_::kSplitWarps;
      constexpr int NG = (TBM / 8) / SW;                   // groups per warp, handled four at a time
      const int sw = warp - C_::kSplitWarp0, r = lane >> 2, q = lane & 3;
      const int xin = (r * RB >> 7) & (RB / 16 - 1);       // swizzle XOR terms of row r in the two layouts
      const int xout = (r * RH >> 7) & (RH / 16 - 1);
      (void)et;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int kb = 0; kb < nkb; ++kb, ++kbg) {
          const int s = (int)(kbg % kStages);
          mbar_wait(&full_bar[s], (uint32_t)((kbg / kStages) & 1));
          uint8_t* base = sA + s * kStageBytesA;
#pragma unroll
          for (int i0 = 0; i0 < NG; i0 += 4) {
          float4 v[4][TBK == 32 ? 2 : 1];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint8_t* gp = base + (sw + SW * (i0 + i)) * GB + r * RB;
            if constexpr (TBK == 32) {
              v[i][0] = *reinterpret_cast<const float4*>(gp + (((2 * q) ^ xin) << 4));
              v[i][1] = *reinterpret_cast<const float4*>(gp + (((2 * q + 1) ^ xin) << 4));
            } else {
              v[i][0] = *reinterpret_cast<const float4*>(gp + ((q ^ xin) << 4));
            }
          }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            uint8_t* gp = base + (sw + SW * (i0 + i)) * GB + r * RH;
            uint32_t hi[TBK == 32 ? 4 : 2], lo[TBK == 32 ? 4 : 2];
#pragma unroll
            for (int j = 0; j < (TBK == 32 ? 2 : 1); ++j) {
              const float4 x = v[i][j];
              const uint32_t h0 = bd_pack_bf16(x.x, x.y), h1 = bd_pack_bf16(x.z, x.w);
              hi[2 * j] = h0;
              hi[2 * j + 1] = h1;
              lo[2 * j] = lo[2 * j + 1] = 0u;
              if constexpr (MODE == BD_TC_BF16X3) {
                lo[2 * j] = bd_pack_bf16(x.x - __uint_as_float(h0 << 16), x.y - __uint_as_float(h0 & 0xffff0000u));
                lo[2 * j + 1] = bd_pack_bf16(x.z - __uint_as_float(h1 << 16), x.w - __uint_as_float(h1 & 0xffff0000u));
              }
            }
            if constexpr (TBK == 32) {
              uint8_t* dst = gp + ((q ^ xout) << 4);
              *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
              if constexpr (MODE == BD_TC_BF16X3) *reinterpret_cast<uint4*>(dst + 8 * RH) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            } else {
              uint8_t* dst = gp + (((q >> 1) ^ xout) << 4) + ((q & 1) << 3);
              *reinterpret_cast<uint2*>(dst) = make_uint2(hi[0], hi[1]);
              if constexpr (MODE == BD_TC_BF16X3) *reinterpret_cast<uint2*>(dst + 8 * RH) = make_uint2(lo[0], lo[1]);
            }
          }
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> UMMA reads
          mbar_arrive(&conv_bar[s]);
        }
      }
    } else {
    // ===== operand splitter (3xTF32): x -> tf32(x) in place, x - tf32(x) into the lo half of the stage =====
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      for (int kb = 0; kb < nkb; ++kb, ++kbg) {
        const int s = (int)(kbg % kStages);
        mbar_wait(&full_bar[s], (uint32_t)((kbg / kStages) & 1));
        auto split = [&](uint8_t* base, int tile_bytes) {
          float4* hi = reinterpret_cast<float4*>(base);
          float4* lo = reinterpret_cast<float4*>(base + tile_bytes);
#pragma unroll 4
          for (int i = et; i < tile_bytes / 16; i += 128) {
            const float4 x = hi[i];
            const float4 h = make_float4(bd_tf32_rna(x.x), bd_tf32_rna(x.y), bd_tf32_rna(x.z), bd_tf32_rna(x.w));
            hi[i] = h;
            lo[i] = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
          }
        };
        split(sA + s * kStageBytesA, kTileBytesA);
        split(sB + s * kStageBytesB, kTileBytesB);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> UMMA reads
        mbar_arrive(&conv_bar[s]);
      }
    }
    }
  } else if (warp >= C_::kEpiWarp0) {
    // ===== epilogue warps: TMEM lane quarter = warp % 4, column group = (warp - first) / 4 =====
    const int quarter = warp & 3, ew = warp - C_::kEpiWarp0, grp = ew >> 2;
    const int cbase = kTileSplit ? 0 : grp * WC;
    const bool row_stats = d.stats_out && d.stat_mod != 1;
    const bool vec = bd_epi_vec_ok(d);
    const int fast = epi_fast_id(d, vec, row_stats);
    constexpr int LDT = WC + 4;
    float* stage = staging + (size_t)ew * 32 * LDT;
    RowInfo* rinfo = reinterpret_cast<RowInfo*>(((uintptr_t)(tmem_slot + 4) + 31) & ~(uintptr_t)31) + ew * 32;
    int tcount = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
      if (kTileSplit && tcount % kPGroups != grp) continue;
      int b, i0s, i1s, n0;
      decode(tile, b, i0s, i1s, n0);
      const int a = tcount % kNAcc;
      const int r = quarter * 32 + lane;
      const int i0 = i0s + (r & (g.R0 - 1)), i1 = i1s + (r >> g.log2R0);
      const bool row_ok = i0 < d.I0 && i1 < d.I1;
      const long long m = ((long long)b * d.I1 + i1) * d.I0 + i0;
      EpiRow er;
      er.obase = 0; er.i0 = 0; er.rb_row = 0; er.e_mean = 0.f; er.e_rstd = 1.f;
      if (row_ok) {                                // (b, i1, i0) are known from the tile: no divisions for the offset
        er.i0 = i0;
        er.obase = (long long)b * d.os_b + (long long)i1 * d.os_1 +
                   (long long)(d.convt ? 4 * i0 - (d.convt == 1 ? 2 : 0) : i0) * d.os_0;
        if (d.rowbias) er.rb_row = (int)((unsigned)m % (unsigned)d.rowbias_period);
        if (d.e_stats) {
          const int sl = bd_stat_slab(d, m);
          er.e_mean = __ldg(d.e_stats + 2 * (size_t)sl);
          er.e_rstd = __ldg(d.e_stats + 2 * (size_t)sl + 1);
        }
      }
      const int my_slab = (d.stats_out && row_ok) ? bd_stat_slab(d, m) : -1;
      float ssum = 0.f, ssq = 0.f;
      if (d.resid && row_ok && !d.convt && !d.oc_split) {
        // this lane's row of the residual operand (one 128-byte line for the warp's column range): start it on
        // its way from HBM to L2 now, the epilogue reads it after the accumulator wait
        const int c0 = n0 + cbase;
        if (c0 < d.N) {
          const float* pf = d.resid + er.obase + (d.act == BD_ACT_GLU ? c0 >> 1 : c0);
          asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
        }
      }
      // a 96 / 192 / 256-column tile is finished in chunks of CHW columns (one staging buffer serves them all)
#pragma unroll 1
      for (int ch = 0; ch < NCH; ++ch) {
      const int n0h = n0 + CHW * ch;
      if (ch == 0) {
        mbar_wait_relaxed(&tmem_full[a], (uint32_t)((tcount / kNAcc) & 1));
        tcgen05_fence_after();
      } else {
        __syncwarp();                              // the staging rows of the previous chunk have been consumed
      }
      const bool last_chunk = ch == NCH - 1;
      const uint32_t acc = tmem_base + (uint32_t)(a * TBN + CHW * ch + cbase) + ((uint32_t)(quarter * 32) << 16);
      if (vec) {
        rinfo[lane].obase = er.obase;
        rinfo[lane].i0 = row_ok ? er.i0 : -1;
        rinfo[lane].rb_row = er.rb_row;
        rinfo[lane].e_mean = er.e_mean;
        rinfo[lane].e_rstd = er.e_rstd;
        for (int c0 = 0; c0 < WC; c0 += CW) {
          if (n0h + cbase + c0 >= d.N) break;
          uint32_t v[CW];
          if constexpr (CW == 32) tmem_ld32(acc + c0, v); else tmem_ld16(acc + c0, v);
#pragma unroll
          for (int j = 0; j < CW; j += 4)
            *reinterpret_cast<float4*>(stage + lane * LDT + c0 + j) =
                make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                            __uint_as_float(v[j + 3]));
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0 && last_chunk) mbar_arrive(&tmem_empty[a]);   // accumulator is free for tile i+2 while we finish tile i
        if (fast >= 0) {
          const uint32_t st_s = smem_u32(stage), ri_s = smem_u32(rinfo);
          const int n0w = n0h + cbase;
          constexpr int FRB = kPGroups >= 4 ? 2 : 4;
          switch (fast) {
            case 0: epi_fast_rows<BD_ACT_NONE, false, false, false, false, WC, FRB>(d, st_s, ri_s, lane, n0w, ssum, ssq); break;
            case 1: epi_fast_rows<BD_ACT_NONE, false, true, false, false, WC, FRB>(d, st_s, ri_s, lane, n0w, ssum, ssq); break;
            case 2: epi_fast_rows<BD_ACT_GELU, false, false, false, false, WC, FRB>(d, st_s, ri_s, lane, n0w, ssum, ssq); break;
            case 3: epi_fast_rows<BD_ACT_GLU, false, false, false, false, WC, FRB>(d, st_s, ri_s, lane, n0w, ssum, ssq); break;
            case 4: epi_fast_rows<BD_ACT_GLU, true, true, false, false, WC, FRB>(d, st_s, ri_s, lane, n0w, ssum, ssq); break;
            case 5: epi_fast_rows<BD_ACT_GLU, false, false, true, false, WC, FRB>(d, st_s, ri_s, lane, n0w, ssum, ssq); break;
            default: epi_fast_rows<BD_ACT_GELU, false, false, false, true, WC, FRB>(d, st_s, ri_s, lane, n0w, ssum, ssq); break;
          }
          __syncwarp();
        } else {
        constexpr int CG = WC / 4 < 32 ? WC / 4 : 32;
        constexpr int RPI = 32 / CG;
        constexpr int RB = kPGroups >= 4 ? 2 : 4;
        const int cg = lane % CG, rsub = lane / CG;
        const int n = n0h + cbase + 4 * cg;
        const bool col_ok = n < d.N;
        EpiCol ecol;
        if (col_ok) ecol = bd_epi_cols4(d, n);
        for (int it = 0; it < 32 / RPI; it += RB) {
          EpiRow row[RB];
          EpiMem mem[RB];
          bool ok[RB];
#pragma unroll
          for (int u = 0; u < RB; ++u) {
            const int rloc = (it + u) * RPI + rsub;
            const uint32_t ra = smem_u32(&rinfo[rloc]);
            uint32_t w0, w1, w2, w3, w4, w5;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "r"(ra));
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(w4), "=r"(w5) : "r"(ra + 16));
            row[u].obase = (long long)(((unsigned long long)w1 << 32) | w0);
            row[u].i0 = (int)w2;
            row[u].rb_row = (int)w3;
            row[u].e_mean = __uint_as_float(w4);
            row[u].e_rstd = __uint_as_float(w5);
            ok[u] = row[u].i0 >= 0 && col_ok;
            if (ok[u]) mem[u] = bd_epi_fetch4(d, row[u], ecol);
          }
#pragma unroll
          for (int u = 0; u < RB; ++u) {
            const int rloc = (it + u) * RPI + rsub;
            float rs = 0.f, rq = 0.f;
            if (ok[u]) {
              const float4 acc4 = *reinterpret_cast<const float4*>(stage + rloc * LDT + 4 * cg);
              bd_epi_finish4(d, row[u], ecol, acc4, mem[u], rs, rq);
            }
            if (row_stats) {
              __syncwarp();
              *reinterpret_cast<float2*>(stage + rloc * LDT + 2 * cg) = make_float2(rs, rq);
            } else {
              ssum += rs;
              ssq += rq;
            }
          }
        }
        if (row_stats) {
          __syncwarp();
          float rs = 0.f, rq = 0.f;
#pragma unroll
          for (int c = 0; c < CG; ++c) {
            const float2 t = *reinterpret_cast<const float2*>(stage + lane * LDT + 2 * c);
            rs += t.x;
            rq += t.y;
          }
          if (my_slab >= 0) {
            atomicAdd(&d.stats_out[2 * (size_t)my_slab], (double)rs);
            atomicAdd(&d.stats_out[2 * (size_t)my_slab + 1], (double)rq);
          }
        }
        __syncwarp();   // staging rows are rewritten by the next tile
        }
      } else {
        for (int c0 = 0; c0 < WC; c0 += CW) {
          if (n0h + cbase + c0 >= d.N) break;
          uint32_t v[CW];
          if constexpr (CW == 32) tmem_ld32(acc + c0, v); else tmem_ld16(acc + c0, v);
          if (row_ok) {
#pragma unroll
            for (int j = 0; j < CW; ++j) {
              const int n = n0h + cbase + c0 + j;
              if (n < d.N) {
                float st;
                if (bd_epi_apply(d, er, n, __uint_as_float(v[j]), __uint_as_float(v[(j + 1) % CW]), st)) {
                  ssum += st;
                  ssq = fmaf(st, st, ssq);
                }
              }
            }
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0 && last_chunk) mbar_arrive(&tmem_empty[a]);
      }
      }   // chunk
      if (!vec && row_stats && row_ok) {       // the row's sums over every chunk
        atomicAdd(&d.stats_out[2 * (size_t)my_slab], (double)ssum);
        atomicAdd(&d.stats_out[2 * (size_t)my_slab + 1], (double)ssq);
      }
      if (d.stats_out && d.stat_mod == 1) {   // one slab per tile (host guarantee): one atomic pair per warp
        const double ds = bd_warp_sum_d((double)ssum), dq = bd_warp_sum_d((double)ssq);
        if (lane == 0) {
          const int sl = bd_stat_slab(d, (long long)b * d.I1 * d.I0 + i0s);
          atomicAdd(&d.stats_out[2 * (size_t)sl], ds);
          atomicAdd(&d.stats_out[2 * (size_t)sl + 1], dq);
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tcgen05_dealloc(tmem_base, kTmemCols);
  }
}

// ---- host side ------------------------------------------------------------------------------------------
template <int TBK, int TBN, int MODE, bool ATM = false>
int launch_tc_persist(const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st) {
  using C_ = PCfg<TBK, TBN, MODE, ATM>;
  alignas(64) CUtensorMap map_a, map_b, map_b_lo;
  const long long s0 = d.xs_0, s1 = d.J1 > 1 ? d.xs_1 : s0 * d.J0, sb = items > 1 ? d.xs_b : s1 * d.J1;
  constexpr int ES = C_::kDirect ? 2 : 4;            // bytes per element of the A tensor
  cuuint64_t adim[5] = {(cuuint64_t)d.Cin, (cuuint64_t)d.J0, (cuuint64_t)d.J1, (cuuint64_t)items, 1};
  cuuint64_t astr[4] = {(cuuint64_t)s0 * ES, (cuuint64_t)s1 * ES, (cuuint64_t)sb * ES, 0};
  cuuint32_t abox[5] = {(cuuint32_t)TBK, (cuuint32_t)g.R0, (cuuint32_t)g.R1, 1, 1};
  int arank = 4;
  if (g.stride4) {
    arank = 5;
    adim[1] = 4; adim[2] = (cuuint64_t)d.J0 / 4; adim[3] = (cuuint64_t)d.J1; adim[4] = (cuuint64_t)items;
    astr[0] = (cuuint64_t)s0 * ES; astr[1] = (cuuint64_t)s0 * 4 * ES; astr[2] = (cuuint64_t)s1 * ES; astr[3] = (cuuint64_t)sb * ES;
    abox[1] = 1; abox[2] = (cuuint32_t)g.R0; abox[3] = (cuuint32_t)g.R1; abox[4] = 1;
  }
  cuuint64_t bdim[2] = {(cuuint64_t)d.K, (cuuint64_t)d.N};
  cuuint32_t bbox[2] = {(cuuint32_t)TBK, (cuuint32_t)TBN};
  bool ok = encode_tensor_map(&map_a, d.x, arank, adim, astr, abox, TBK * ES, C_::kDirect);
  if constexpr (C_::kB16) {
    cuuint64_t bstr[1] = {(cuuint64_t)d.K * 2};
    ok = ok && encode_tensor_map(&map_b, d.w16_hi, 2, bdim, bstr, bbox, TBK * 2, true);
    ok = ok && encode_tensor_map(&map_b_lo, MODE == BD_TC_BF16X3 ? d.w16_lo : d.w16_hi, 2, bdim, bstr, bbox, TBK * 2, true);
  } else {
    cuuint64_t bstr[1] = {(cuuint64_t)d.K * 4};
    ok = ok && encode_tensor_map(&map_b, d.w, 2, bdim, bstr, bbox, TBK * 4);
    map_b_lo = map_b;
  }
  if (!ok) {
    bd_set_error("bd_conv_gemm_tc: TMA tensor map encoding failed (M=%d N=%d K=%d Cin=%d J0=%d J1=%d)", d.M, d.N, d.K,
                 d.Cin, d.J0, d.J1);
    return BD_ERR_CUDA;
  }
  // per device: the opt-in shared-memory size is an attribute of the function ON a device, and the persistent
  // grid is one CTA per SM of the device the launch goes to
  static int sms_of[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) {
    bd_set_error("bd_conv_gemm_tc: device ordinal %d out of range", dev);
    return BD_ERR_ARG;
  }
  if (!sms_of[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv_gemm_tc_persist_kernel<TBK, TBN, MODE, ATM>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, C_::kSmemBytes);
    if (e != cudaSuccess) {
      bd_set_error("bd_conv_gemm_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return BD_ERR_CUDA;
    }
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    sms_of[dev] = n;
  }
  const int sms = sms_of[dev];
  const int ntn = (d.N + TBN - 1) / TBN;
  const long long ntiles = (long long)items * g.blocks1 * g.blocks0 * ntn;
  const int grid = (int)(ntiles < sms ? ntiles : sms);
  conv_gemm_tc_persist_kernel<TBK, TBN, MODE, ATM><<<grid, C_::kThreads, C_::kSmemBytes, st>>>(map_a, map_b, map_b_lo, d,
                                                                                              g, (int)ntiles, ntn);
  return bd_check_launch("conv_gemm_tc_persist_kernel");
}

// every tile width up to 192 of one (k-block depth, arithmetic, A operand location) triple; the 96 / 192-column
// tiles exist for the strict mode only (tile_width in gemm_tc.cu)
template <int TBK, int MODE, bool ATM = false>
int launch_tc_width(int tbn, const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st) {
  switch (tbn) {
    case 16: return launch_tc_persist<TBK, 16, MODE, ATM>(d, g, items, st);
    case 32: return launch_tc_persist<TBK, 32, MODE, ATM>(d, g, items, st);
    case 64: return launch_tc_persist<TBK, 64, MODE, ATM>(d, g, items, st);
    case 128: return launch_tc_persist<TBK, 128, MODE, ATM>(d, g, items, st);
    default: break;
  }
  if constexpr (MODE == BD_TC_BF16X3) {
    if (tbn == 96) return launch_tc_persist<TBK, 96, MODE, ATM>(d, g, items, st);
    if (tbn == 192) return launch_tc_persist<TBK, 192, MODE, ATM>(d, g, items, st);
  }
  bd_set_error("bd_conv_gemm_tc: no kernel for tile width %d", tbn);
  return BD_ERR_ARG;
}

}  // namespace
