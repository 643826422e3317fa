// Development probe: resident blocks per SM of both K10 instantiations with the driver's default
// shared-memory carve-out, and their registers (profiles/r07_k10_four_blocks.md).
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I../../include tb3_occupancy.cu -o tb3_occupancy
#include "../../advanced-hpc-lbm_b200/csrc/lbm_tb3.cuh"
#include <cstdio>
#include <cstdlib>
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1);} } while (0)

template <bool STRICT>
static int report(const char* name) {
  const void* fn = (const void*)lbm::lbm_step3_tb<STRICT>;
  CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(lbm::Tb3Smem)));
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, fn));
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, LBM_TB2_THREADS, sizeof(lbm::Tb3Smem)));
  printf("%s: %d registers, %zu B static + %zu B dynamic shared memory, %d blocks of %d threads per SM "
         "(LBM_TB3_MIN_BLOCKS %d)\n", name, fa.numRegs, fa.sharedSizeBytes, sizeof(lbm::Tb3Smem), per_sm,
         LBM_TB2_THREADS, LBM_TB3_MIN_BLOCKS);
  return per_sm == LBM_TB3_MIN_BLOCKS ? 0 : 1;
}

int main() {
  int smem_sm = 0;
  CK(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, 0));
  printf("shared memory per SM: %d B\n", smem_sm);
  const int bad = report<false>("lbm_step3_tb<false>") + report<true>("lbm_step3_tb<true>");
  return bad ? 1 : 0;
}
