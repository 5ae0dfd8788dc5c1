// K3/K4/K7 (tensor-core arm): the BD_TC_BF16X3 instantiations that split the fp32 A tile in place in shared memory:
// the 256-column tiles, whose accumulators leave no tensor memory for the operand, and every narrower width for
// comparison with the tensor-memory path (BD_TC_SMEM_A=1).  A separate translation unit so that the two families
// compile in parallel.
#include "gemm_tc_impl.cuh"

int bd_tc_launch_bf16x3_smem_a(int tbk, int tbn, const bd_gemm_desc& d, const TileGeom& g, int items, cudaStream_t st) {
  if (tbk == 32)
    return tbn == 256 ? launch_tc_persist<32, 256, BD_TC_BF16X3>(d, g, items, st) : launch_tc_width<32, BD_TC_BF16X3>(tbn, d, g, items, st);
  return tbn == 256 ? launch_tc_persist<16, 256, BD_TC_BF16X3>(d, g, items, st) : launch_tc_width<16, BD_TC_BF16X3>(tbn, d, g, items, st);
}
