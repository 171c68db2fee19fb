// Pieces shared by the LSTM recurrence (lstm_sm100.cu) and its backward (lstm_train_sm100.cu): the cluster layout of a
// hidden size, the 16-byte st.async message and the fast gate activations.
#pragma once
#include <cuda_bf16.h>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"

namespace svsk {

constexpr int kLstmMaxThreads = 256;

__device__ __forceinline__ void st_async_v4(uint32_t cluster_addr, float a, float b, float c, float d, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(cluster_addr),
               "f"(a), "f"(b), "f"(c), "f"(d), "r"(cluster_mbar)
               : "memory");
}

// Gate activations on the critical path of every step: ex2.approx / rcp.approx forms, absolute error ~1e-6 (the fp32
// parity tolerance is 2e-4), a third of the dependent-instruction chain of expf / tanhf.
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return rcp_fast(1.f + ex2_fast(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_fast(float x) { return fmaf(-2.f, rcp_fast(1.f + ex2_fast(2.8853900817779268f * x)), 1.f); }

// H -> (CTAs per cluster, units per CTA, column segments per unit, segment length); false when H has no layout here.
inline bool lstm_layout(int H, int* NC, int* U, int* CS, int* L) {
  if (H < 4 || H > 256 || H % 4) return false;
  int cs = 1;
  while (H / cs > 32 || H % cs) {
    cs *= 2;
    if (cs > 8) return false;
  }
  if (H % (4 * cs)) return false;  // segments hold whole quads of units (16-byte messages)
  for (int nc = 1; nc <= 8; nc *= 2) {
    if (H % (4 * nc) || H / nc > 32) continue;
    *NC = nc;
    *U = H / nc;
    *CS = cs;
    *L = H / cs;
    return true;
  }
  return false;
}

// Launches kernel<<<B * ndir * NC CTAs in clusters of NC>>>(args).
template <typename Args>
inline int launch_cluster(void (*kernel)(Args), const Args& a, int ctas, int nc, int threads, cudaStream_t st, const char* what) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)ctas);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)nc;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, a);
  if (e != cudaSuccess) return fail((int)e, "%s: launch: %s", what, cudaGetErrorString(e));
  return 0;
}

}  // namespace svsk
