// rt_adaptive.cu — per-pixel state of rt_render_adaptive between the passes of the error-map path tracer.
//
// A pass traces a list of pixels (pass 0: every pixel) with launch_pt_warp_err, which leaves the pass mean
// m_p and its squared standard error SE_p^2 per list entry.  Here, per listed pixel:
//   combine   sum_m += m_p, sum_v += SE_p^2, passes += 1 (fp32, in pass order)
//   select    the pixel is traced again if its relative error e = max_c sqrt(sum_v) / P / max(sum_m / P, floor)
//             is above the target and it has passes left; the next list holds those pixels in ascending order
//             (the order decides which pixels share a task, so the compaction is deterministic: per-tile
//             counts, one ordered scan of the counts, then every tile writes its pixels at its offset)
//   final     mean = sum_m / P, SE = sqrt(sum_v) / P, samples = P * S^2 for every pixel
#include <algorithm>

#include "rt_launch.h"

#define RT_AD_THREADS 256
#define RT_AD_ITEMS 8                              // consecutive list entries per thread
#define RT_AD_TILE (RT_AD_THREADS * RT_AD_ITEMS)

// exclusive block-wide scan of one int per thread (RT_AD_THREADS threads); returns the block total in *total
__device__ int block_exclusive_scan(int v, int* total) {
  __shared__ int warp_sums[RT_AD_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  if (lane == 31) warp_sums[warp] = x;
  __syncthreads();
  int before = 0, all = 0;
  for (int w = 0; w < RT_AD_THREADS / 32; ++w) {
    if (w < warp) before += warp_sums[w];
    all += warp_sums[w];
  }
  __syncthreads();
  *total = all;
  return before + x - v;
}

__device__ bool adaptive_wants_more(const float* sm, const float* sv, int passes, float target, float floor_) {
  const float P = (float)passes;
  float e = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float mean = __fdiv_rn(sm[c], P), se = __fdiv_rn(__fsqrt_rn(sv[c]), P);
    e = fmaxf(e, __fdiv_rn(se, fmaxf(mean, floor_)));
  }
  return e > target;
}

__global__ void __launch_bounds__(RT_AD_THREADS)
k_adaptive_combine(const int32_t* list, int n, const float* em, const float* ev, int pass, bool select, float target, float floor_,
                   float* sum_m, float* sum_v, int32_t* n_pass, uint8_t* flags, int32_t* block_counts) {
  const int first = blockIdx.x * RT_AD_TILE + threadIdx.x * RT_AD_ITEMS;
  int count = 0;
  for (int k = 0; k < RT_AD_ITEMS; ++k) {
    const int i = first + k;
    if (i >= n) break;
    const int px = list ? list[i] : i;
    float* sm = sum_m + 3 * (size_t)px;
    float* sv = sum_v + 3 * (size_t)px;
    int P;
    if (pass == 0) {
      for (int c = 0; c < 3; ++c) { sm[c] = em[3 * (size_t)i + c]; sv[c] = ev[3 * (size_t)i + c]; }
      P = 1;
    } else {
      for (int c = 0; c < 3; ++c) { sm[c] = __fadd_rn(sm[c], em[3 * (size_t)i + c]); sv[c] = __fadd_rn(sv[c], ev[3 * (size_t)i + c]); }
      P = n_pass[px] + 1;
    }
    n_pass[px] = P;
    const bool more = select && adaptive_wants_more(sm, sv, P, target, floor_);
    flags[i] = more ? 1 : 0;
    count += more;
  }
  int total;
  block_exclusive_scan(count, &total);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// one block: block_counts[0 .. nb) -> exclusive offsets, the sum -> *d_count
__global__ void __launch_bounds__(RT_AD_THREADS) k_adaptive_offsets(int32_t* block_counts, int nb, int32_t* d_count) {
  int carry = 0;
  for (int base = 0; base < nb; base += RT_AD_THREADS) {
    const int i = base + threadIdx.x;
    const int v = i < nb ? block_counts[i] : 0;
    int total;
    const int ex = block_exclusive_scan(v, &total);
    if (i < nb) block_counts[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) *d_count = carry;
}

__global__ void __launch_bounds__(RT_AD_THREADS)
k_adaptive_scatter(const int32_t* list, int n, const uint8_t* flags, const int32_t* offsets, int32_t* next_list) {
  const int first = blockIdx.x * RT_AD_TILE + threadIdx.x * RT_AD_ITEMS;
  int count = 0;
  for (int k = 0; k < RT_AD_ITEMS && first + k < n; ++k) count += flags[first + k];
  int total;
  int at = offsets[blockIdx.x] + block_exclusive_scan(count, &total);
  for (int k = 0; k < RT_AD_ITEMS && first + k < n; ++k) {
    const int i = first + k;
    if (flags[i]) next_list[at++] = list ? list[i] : i;
  }
}

__global__ void k_adaptive_final(const float* sum_m, const float* sum_v, const int32_t* n_pass, int spp, int n, float* rgb, float* err,
                                 int32_t* samples) {
  for (int px = blockIdx.x * blockDim.x + threadIdx.x; px < n; px += gridDim.x * blockDim.x) {
    const int P = n_pass[px];
    const float fp = (float)P;
    for (int c = 0; c < 3; ++c) {
      rgb[3 * (size_t)px + c] = __fdiv_rn(sum_m[3 * (size_t)px + c], fp);
      if (err) err[3 * (size_t)px + c] = __fdiv_rn(__fsqrt_rn(sum_v[3 * (size_t)px + c]), fp);
    }
    if (samples) samples[px] = P * spp;
  }
}

cudaError_t launch_adaptive_combine(const ErrArgs& e, int pass, int max_passes, float target, float floor_, float* sum_m, float* sum_v,
                                    int32_t* n_pass, uint8_t* flags, int32_t* block_counts, int32_t* d_count, int32_t* next_list, int n_pixels,
                                    cudaStream_t st, LaunchInfo* info) {
  const int n = e.pix_list ? (int)e.n_list : n_pixels;
  const bool select = pass + 1 < max_passes;
  const int nb = (n + RT_AD_TILE - 1) / RT_AD_TILE;
  if (nb == 0) return cudaMemsetAsync(d_count, 0, sizeof(int32_t), st);
  k_adaptive_combine<<<nb, RT_AD_THREADS, 0, st>>>(e.pix_list, n, e.err_mean, e.err_var, pass, select, target, floor_, sum_m, sum_v,
                                                   n_pass, flags, block_counts);
  k_adaptive_offsets<<<1, RT_AD_THREADS, 0, st>>>(block_counts, nb, d_count);
  k_adaptive_scatter<<<nb, RT_AD_THREADS, 0, st>>>(e.pix_list, n, flags, block_counts, next_list);
  if (info) info->n_launches += 3;
  return cudaGetLastError();
}

cudaError_t launch_adaptive_final(const float* sum_m, const float* sum_v, const int32_t* n_pass, int spp, int n_pixels, float* rgb, float* err,
                                  int32_t* samples, cudaStream_t st, LaunchInfo* info) {
  const int blocks = std::min((n_pixels + 255) / 256, 148 * 16);
  if (blocks == 0) return cudaSuccess;
  k_adaptive_final<<<blocks, 256, 0, st>>>(sum_m, sum_v, n_pass, spp, n_pixels, rgb, err, samples);
  if (info) info->n_launches += 1;
  return cudaGetLastError();
}
