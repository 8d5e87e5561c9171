// rt_kernels_f32.cu — float instantiations (multiply-add fusion allowed) + the warp-cooperative
// path tracer, which exists in fp32 only.
#include <cstdlib>

#include "rt_warp.cuh"
#include "rt_warp_bvh.cuh"
#include "rt_resolve_f32.cuh"

template <> cudaError_t launch_resolve<float>(const SceneView<float>& sc, const RenderArgs& a, cudaStream_t st, LaunchInfo* info) {
  return launch_resolve_f32(sc, a, st, info);
}
template cudaError_t launch_pt_mega<float>(const SceneView<float>&, const RenderArgs&, cudaStream_t, LaunchInfo*);
template cudaError_t launch_probe<float>(const SceneView<float>&, const RenderArgs&, const ProbeArgs&, cudaStream_t);

cudaError_t launch_pt_warp(const SceneView<float>& sc, const RenderArgs& a, cudaStream_t st, int sm_count,
                           LaunchInfo* info, const char** why_not, int n_nodes, int n_prims, int tree_depth) {
  if (sc.accel) return launch_pt_warp_bvh(sc, a, st, sm_count, info, why_not, n_nodes, n_prims, tree_depth);  // sphere hierarchy: its own schedule
  return launch_pt_warp_impl(sc, a, st, sm_count, info, why_not);
}

cudaError_t launch_pt_warp_err(const SceneView<float>& sc, const RenderArgs& a, const ErrArgs& e, cudaStream_t st, int sm_count,
                               LaunchInfo* info, const char** why_not, int n_nodes, int n_prims, int tree_depth) {
  if (sc.accel) return launch_pt_warp_bvh<true>(sc, a, st, sm_count, info, why_not, n_nodes, n_prims, tree_depth, e);
  return launch_pt_warp_impl<true>(sc, a, st, sm_count, info, why_not, e);
}

// FP32 FMA throughput probe: the denominator of the roofline this path is bound by.
__global__ void __launch_bounds__(256) k_ffma(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
#pragma unroll 1
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

cudaError_t launch_ffma(float* out, int blocks, int iters, cudaStream_t st) {
  k_ffma<<<blocks, 256, 0, st>>>(out, iters, 0.999f, 0.001f);
  return cudaGetLastError();
}
