// K3/K4/K7 (tensor-core arm): dispatch of an implicit-GEMM descriptor to the persistent tcgen05 kernel
// (gemm_tc_impl.cuh), and the TF32 / 3xTF32 instantiations.  The bf16-operand families are compiled in
// gemm_tc_b16x3.cu / gemm_tc_b16.cu.
#include "gemm_tc_impl.cuh"

int bd_tc_launch_bf16x3(int tbk, int tbn, const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st);
int bd_tc_launch_bf16(int tbk, int tbn, const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st);
int bd_tc_launch_bf16d(int tbk, int tbn, const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st);

namespace {
int pow2_ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}
}  // namespace

// eligibility: unit-stride implicit GEMM, channels-last, big enough to fill tensor-core tiles
bool bd_conv_gemm_tc_eligible(const bd_gemm_desc& d) {
  if (d.a_mode != BD_A_NONE || d.xs_c != 1 || d.m1 != 1) return false;
  if (!(d.m0 == 1 || (d.m0 == 4 && d.J0 % 4 == 0))) return false;
  if (d.Cin % 16 != 0 || d.N < 16 || d.K < 16 || d.M < 128 || d.taps > BD_MAX_TAPS) return false;
  if (d.x_bf16) {   // bf16 A tensor: TMA strides are multiples of 16 bytes = 8 elements, 64-element k-blocks
    if (d.math != BD_MATH_BF16 || d.Cin % 64 != 0) return false;
    if (d.xs_0 % 8 != 0 || (d.J1 > 1 && d.xs_1 % 8 != 0) || d.xs_b % 8 != 0) return false;
  }
  if (d.xs_0 % 4 != 0 || (d.J1 > 1 && d.xs_1 % 4 != 0) || d.xs_b % 4 != 0) return false;
  if (((uintptr_t)d.x & 15) || ((uintptr_t)d.w & 15)) return false;
  if (d.math == BD_MATH_BF16X3 || d.math == BD_MATH_BF16) {   // pre-split bf16 weight planes [N, K]
    if (!d.w16_hi || ((uintptr_t)d.w16_hi & 15) || d.K % 8 != 0) return false;
    if (d.math == BD_MATH_BF16X3 && (!d.w16_lo || ((uintptr_t)d.w16_lo & 15))) return false;
  }
  if (d.stats_out && d.stat_mod == 1 && !(d.I1 == 1 && d.I0 == d.stat_div)) return false;
  return true;
}

namespace {

TileGeom tile_geometry(const bd_gemm_desc& d) {
  TileGeom g;
  g.R0 = (d.I0 >= 128 || d.I1 == 1) ? 128 : (pow2_ceil(d.I0) > 128 ? 128 : pow2_ceil(d.I0));
  g.R1 = 128 / g.R0;
  g.log2R0 = 0;
  while ((1 << g.log2R0) < g.R0) ++g.log2R0;
  g.blocks0 = (d.I0 + g.R0 - 1) / g.R0;
  g.blocks1 = (d.I1 + g.R1 - 1) / g.R1;
  g.stride4 = d.m0 == 4;
  g.cpb = 0;
  return g;
}

// Tile width of an eligible descriptor (BD_TC_NO_EXACT is read per call so that both choices can be compared in
// one process).  256-column tiles for the long-K GEMMs whose epilogue has a compile-time
// form: one 128x256x8 MMA reads 12 KB of shared memory for the work of two 128x128x8 MMAs (16 KB) -- the tf32
// kernel is operand-bandwidth-bound -- unless the halved tile count quantises badly over the SMs (short M, N = 512:
// 2.3 waves instead of 4.5).
int tile_width(const bd_gemm_desc& d, const TileGeom& g) {
  static const bool wide_ok = getenv("BD_TC_NO_WIDE") == nullptr;
  static const bool wide_x3 = getenv("BD_TC_NO_WIDE_X3") == nullptr;
  const int items = d.M / (d.I0 * d.I1);
  const bool wide = wide_ok && (d.math != BD_MATH_TF32X3 || wide_x3) && d.N % 256 == 0 &&
                    d.K >= 256 && d.out && !d.convt && !d.oc_split && !d.rowbias && !d.addend && !d.e_stats &&
                    (!d.stats_out || d.stat_mod == 1) && bd_epi_vec_ok(d);
  auto wave_eff = [&](int tile_n) {
    const long long t = (long long)items * g.blocks1 * g.blocks0 * ((d.N + tile_n - 1) / tile_n);
    return (double)t / (double)(((t + 147) / 148) * 148);
  };
  if (wide && wave_eff(256) >= wave_eff(128) - 0.05) return 256;
  const int pow2 = d.N <= 16 ? 16 : d.N <= 32 ? 32 : d.N <= 64 ? 64 : 128;
  // strict mode: 96 / 192-column tiles where the power-of-two ones would pad N by a quarter or more (the N = 96 / 192
  // decoder and DConv layers: a quarter of the MMAs and B traffic, and for 192 one of two A tile loads, saved)
  if (d.math == BD_MATH_BF16X3 && getenv("BD_TC_NO_EXACT") == nullptr) {
    const int exact = (d.N > 64 && d.N <= 96) ? 96 : (d.N > 128 && d.N <= 192) ? 192 : 0;
    if (exact && wave_eff(exact) >= wave_eff(pow2) - 0.05) return exact;
  }
  return pow2;
}

}  // namespace

// k-block depth (floats of K per pipeline stage).  TF32: 32 unless the tile is 256 wide (stage size) or Cin is an odd
// multiple of 16; 3xTF32: 16 (hi/lo stages are twice the size); bf16 families: 32 whenever Cin allows (the fp32 stage
// is split in place, so the stage does not grow).
static int k_block(const bd_gemm_desc& d, int tbn) {
  if (d.x_bf16) return 64;
  if (d.math == BD_MATH_BF16X3 || d.math == BD_MATH_BF16) return d.Cin % 32 == 0 ? 32 : 16;
  return (tbn == 256 || d.math == BD_MATH_TF32X3 || d.Cin % 32 != 0) ? 16 : 32;
}

// 0: the descriptor is not eligible for the tensor-core arm; else 1000 * TBK + TBN of the kernel template it runs
int bd_conv_gemm_tc_tile(const bd_gemm_desc& d) {
  if (!bd_conv_gemm_tc_eligible(d) || d.M % ((long long)d.I0 * d.I1) != 0) return 0;
  const int tbn = tile_width(d, tile_geometry(d));
  return 1000 * k_block(d, tbn) + tbn;
}

int bd_conv_gemm_tc(const bd_gemm_desc* dp, void* stream, int* handled) {
  const bd_gemm_desc& d = *dp;
  *handled = 0;
  if (!bd_conv_gemm_tc_eligible(d)) return BD_OK;
  BD_REQUIRE(d.act != BD_ACT_GLU || d.N % 2 == 0, "bd_conv_gemm: GLU needs even N");
  BD_REQUIRE(d.M % ((long long)d.I0 * d.I1) == 0, "bd_conv_gemm: M not a multiple of I1*I0");
  TileGeom g = tile_geometry(d);
  const int items = d.M / (d.I0 * d.I1);
  const int tbn = tile_width(d, g);
  const int tbk = k_block(d, tbn);
  g.cpb = d.Cin / tbk;
  const cudaStream_t st = (cudaStream_t)stream;
  int rc;
  switch (d.math) {
    case BD_MATH_BF16X3: rc = bd_tc_launch_bf16x3(tbk, tbn, d, g, items, st); break;
    case BD_MATH_BF16:
      rc = d.x_bf16 ? bd_tc_launch_bf16d(tbk, tbn, d, g, items, st) : bd_tc_launch_bf16(tbk, tbn, d, g, items, st);
      break;
    case BD_MATH_TF32X3:
      rc = tbn == 256 ? launch_tc_persist<16, 256, BD_TC_TF32X3>(d, g, items, st)
                      : launch_tc_width<16, BD_TC_TF32X3>(tbn, d, g, items, st);
      break;
    default:
      rc = tbn == 256 ? launch_tc_persist<16, 256, BD_TC_TF32>(d, g, items, st)
           : tbk == 32 ? launch_tc_width<32, BD_TC_TF32>(tbn, d, g, items, st)
                       : launch_tc_width<16, BD_TC_TF32>(tbn, d, g, items, st);
      break;
  }
  *handled = 1;
  return rc;
}
