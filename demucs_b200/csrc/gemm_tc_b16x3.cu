// K3/K4/K7 (tensor-core arm): the BD_TC_BF16X3 instantiations of the persistent tcgen05 implicit-GEMM kernel
// (gemm_tc_impl.cuh): bf16 operands, fp32 accumulation, error-compensated hi/lo split.  Tiles up to 192 columns
// take the split A operand from tensor memory; 256-column tiles (and every width under BD_TC_SMEM_A=1) split it in
// place in shared memory (gemm_tc_b16x3_smem.cu).
#include "gemm_tc_impl.cuh"

int bd_tc_launch_bf16x3_smem_a(int tbk, int tbn, const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st);

int bd_tc_launch_bf16x3(int tbk, int tbn, const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st) {
  if (tbn == 256 || getenv("BD_TC_SMEM_A") != nullptr) return bd_tc_launch_bf16x3_smem_a(tbk, tbn, d, g, items, st);
  return tbk == 32 ? launch_tc_width<32, BD_TC_BF16X3, true>(tbn, d, g, items, st)
                   : launch_tc_width<16, BD_TC_BF16X3, true>(tbn, d, g, items, st);
}
