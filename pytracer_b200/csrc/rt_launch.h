// rt_launch.h — what rt_api.cu (host side of the C-ABI) and the two kernel translation units
// (rt_kernels_f32.cu, rt_kernels_f64.cu) agree on.
#pragma once
#include "rt_device.cuh"

// counters[] slots in device memory (unsigned long long each)
enum { CNT_CLOSEST = 0, CNT_SHADOW = 1, CNT_SAMPLES = 2, CNT_OVERFLOW = 3, CNT_TASK = 4, CNT_SLOTS = 8 };

struct RenderArgs {
  int32_t width, height, S, algorithm;
  DevCamera cam;
  double background[3], onoff[3], ambient[3];
  int32_t num_of_rays, max_depth, rr_limit, rng_mode;
  uint64_t aa_state, aa_inc, pt_state, pt_inc;
  const uint64_t* replay;  // device copy of rt_render_params.replay_states
  int32_t part_mode, part_rank, part_count, out_f64;
  int32_t hit_mode, rows_compact;  // rows_compact: RT_PART_ROWS stores the owned rows densely
  void* out_rgb;           // float or double [H][W][3]
  float* peer_out[RT_MAX_PEERS];  // n_peers > 0: fp32 full-size images of all ranks, every pixel goes to each
  int32_t n_peers, _pad2;
  int32_t* out_hit;        // optional
  unsigned long long* counters;
  JumpTable jump;          // for the jitter stream (aa_inc)
};

// What the error-map instantiations of the warp path tracers read besides RenderArgs (the last kernel
// parameter of every instantiation, so that the others keep their parameter offsets and code)
struct ErrArgs {
  const int32_t* pix_list; // non-null: the task source is this list of full-image pixels (row * width + col)
  long long n_list;        // entries of pix_list
  float* err_mean;         // [entries][3] pass mean of each traced pixel (list entry, or pixel index without a list)
  float* err_var;          // [entries][3] squared standard error of that mean
  int err_bpp;             // batches per pixel slot of a task (32 / G), set by the launcher
  unsigned err_magic;      // multiply-shift magic of x / err_bpp for x < 32
  int32_t estimator;       // RT_ERR_EST_*: how err_store forms SE^2 from the batch sums
};

struct LaunchInfo {
  int32_t n_launches;
  int32_t variant;
};

// Explicitly instantiated for float in rt_kernels_f32.cu and for double in rt_kernels_f64.cu.
template <typename T> cudaError_t launch_resolve(const SceneView<T>& sc, const RenderArgs& a, cudaStream_t st, LaunchInfo* info);
// rt_kernels_f64.cu: fp32 conservative gate + the reference's fp64 decisions (rt_resolve_hybrid.cuh); `co` is
// device scratch of resolve_hybrid_table_bytes() bytes, perspective cameras only
size_t resolve_hybrid_table_bytes(int n_spheres, int n_lights);
cudaError_t launch_resolve_hybrid(const SceneView<double>& sc, const RenderArgs& a, float* co, cudaStream_t st, LaunchInfo* info);
template <typename T> cudaError_t launch_pt_mega(const SceneView<T>& sc, const RenderArgs& a, cudaStream_t st, LaunchInfo* info);
// fp32 only (rt_kernels_f32.cu): the warp-cooperative wavefront path tracer
// (n_nodes / n_prims / tree_depth describe the sphere hierarchy and are read only when sc.accel != 0)
cudaError_t launch_pt_warp(const SceneView<float>& sc, const RenderArgs& a, cudaStream_t st, int sm_count, LaunchInfo* info, const char** why_not,
                           int n_nodes, int n_prims, int tree_depth);
// the same kernels instantiated with per-pixel error accumulation (ERR): no image is stored; every traced
// pixel gets its pass mean (the value launch_pt_warp stores, bit for bit) and squared standard error in
// e.err_mean / e.err_var, indexed by list entry (e.pix_list) or pixel; needs S >= 2 and no partition
cudaError_t launch_pt_warp_err(const SceneView<float>& sc, const RenderArgs& a, const ErrArgs& e, cudaStream_t st, int sm_count,
                               LaunchInfo* info, const char** why_not, int n_nodes, int n_prims, int tree_depth);
// rt_adaptive.cu: fold a pass into the per-pixel sums, then compact the pixels still to trace
cudaError_t launch_adaptive_combine(const ErrArgs& e, int pass, int max_passes, float target, float floor_, float* sum_m, float* sum_v,
                                    int32_t* n_pass, uint8_t* flags, int32_t* block_counts, int32_t* d_count, int32_t* next_list, int n_pixels,
                                    cudaStream_t st, LaunchInfo* info);
cudaError_t launch_adaptive_final(const float* sum_m, const float* sum_v, const int32_t* n_pass, int spp, int n_pixels, float* rgb, float* err,
                                  int32_t* samples, cudaStream_t st, LaunchInfo* info);

// single-stream probes behind rt_trace_rays / rt_intersect / ... (n items, one thread walks them
// in order when a PCG stream is shared, otherwise one thread per item)
struct ProbeArgs {
  int32_t what, n, aux;     // aux: pigment / material index
  const double* in;         // device
  const int32_t* depth;     // device, optional
  double* out;              // device
  rt_hit* hits;             // device
  uint8_t* flags;           // device
  uint64_t* pcg;            // device {state, inc}, updated
  uint32_t* draws;          // device
};
enum { PROBE_TRACE = 0, PROBE_INTERSECT = 1, PROBE_VISIBLE = 2, PROBE_PIGMENT = 3, PROBE_SCATTER = 4,
       PROBE_ONB = 5, PROBE_PCG_DRAW = 6, PROBE_PCG_SEED = 7, PROBE_CAMERA_RAYS = 8, PROBE_CAMERA_UV = 9 };
template <typename T> cudaError_t launch_probe(const SceneView<T>& sc, const RenderArgs& a, const ProbeArgs& p, cudaStream_t st);

// rt_tonemap.cu: HdrImage.average_luminosity's sum and the normalise / clamp / LDR map (hdrimages.py:120-171)
int tonemap_max_blocks();
cudaError_t launch_lum_sum(const float* d_rgb, long long n_pixels, double delta, double* d_partials,
                           unsigned int* d_done, double* d_out, int sm_count, cudaStream_t st);
cudaError_t launch_tone_map(const float* d_rgb, long long n_pixels, int flags, double scale, double gamma, float* d_out_hdr,
                            unsigned char* d_out_ldr, int sm_count, cudaStream_t st);

cudaError_t launch_ffma(float* out, int blocks, int iters, cudaStream_t st);
cudaError_t launch_dfma(double* out, int blocks, int iters, cudaStream_t st);
