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

// relative error e = max_c (sqrt(sum_v) / P) / max(sum_m / P, floor) of a pixel with P passes; never NaN (fmaxf
// drops a NaN operand) and >= 0, so its bit pattern orders like an unsigned int
__device__ __forceinline__ float adaptive_rel_error(const float* sm, const float* sv, int passes, float floor_) {
  const float P = (float)passes;
  float e = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float mean = __fdiv_rn(sm[c], P), se = __fdiv_rn(__fsqrt_rn(sv[c]), P);
    e = fmaxf(e, __fdiv_rn(se, fmaxf(mean, floor_)));
  }
  return e;
}

__device__ bool adaptive_wants_more(const float* sm, const float* sv, int passes, float target, float floor_) {
  return adaptive_rel_error(sm, sv, passes, floor_) > target;
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

// ---- sample-budget mode (rt_render_adaptive_budget): the next pass traces the K pixels of largest e
//   combine   as above, and e of every listed pixel goes to err_e[px] (a pixel keeps its e until traced again)
//   select    key = e > target ? bits(e) : 0 (e >= 0, so bits order like e); C = #keys > 0; K from C, Q and r on
//             the device; the K-th largest key T by a radix select over four 8-bit digits (integer histograms,
//             one block per digit picks the bucket); then every pixel with key > T and the first K - #(key > T)
//             pixels with key == T in index order (ordered tie ranks: per-tile counts, one ordered scan) are
//             flagged and compacted like the threshold mode's flags
__global__ void __launch_bounds__(RT_AD_THREADS)
k_adaptive_combine_budget(const int32_t* list, int n, const float* em, const float* ev, int pass, float floor_, float* sum_m,
                          float* sum_v, int32_t* n_pass, float* err_e) {
  const int i = blockIdx.x * RT_AD_THREADS + threadIdx.x;
  if (i >= n) return;
  const int px = list ? list[i] : i;
  float sm[3], sv[3];
  int P;
  if (pass == 0) {
    for (int c = 0; c < 3; ++c) { sm[c] = em[3 * (size_t)i + c]; sv[c] = ev[3 * (size_t)i + c]; }
    P = 1;
  } else {
    for (int c = 0; c < 3; ++c) {
      sm[c] = __fadd_rn(sum_m[3 * (size_t)px + c], em[3 * (size_t)i + c]);
      sv[c] = __fadd_rn(sum_v[3 * (size_t)px + c], ev[3 * (size_t)i + c]);
    }
    P = n_pass[px] + 1;
  }
  for (int c = 0; c < 3; ++c) { sum_m[3 * (size_t)px + c] = sm[c]; sum_v[3 * (size_t)px + c] = sv[c]; }
  n_pass[px] = P;
  err_e[px] = adaptive_rel_error(sm, sv, P, floor_);
}

__device__ __forceinline__ unsigned budget_key(float e, float target) { return e > target ? __float_as_uint(e) : 0u; }

// histogram of digit `digit` (bits 8 digit .. 8 digit + 7) of the candidate keys whose higher digits equal the prefix
// picked so far; lanes with the same bin are aggregated before the shared atomic
__global__ void __launch_bounds__(RT_AD_THREADS)
k_budget_hist(const float* err_e, int n, float target, int digit, const BudgetSelect* sel, int32_t* hist) {
  __shared__ int h[256];
  if (digit < 3 && sel->k_rem == 0) return;  // K = 0: nothing to select
  const unsigned hi_mask = digit == 3 ? 0u : 0xFFFFFFFFu << (8 * (digit + 1));
  const unsigned want = sel->prefix & hi_mask;
  h[threadIdx.x] = 0;
  __syncthreads();
  for (int base = blockIdx.x * RT_AD_THREADS; base < n; base += gridDim.x * RT_AD_THREADS) {
    const int i = base + threadIdx.x;
    int bin = -1;
    if (i < n) {
      const unsigned key = budget_key(err_e[i], target);
      if (key && (key & hi_mask) == want) bin = (key >> (8 * digit)) & 255;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[bin], __popc(peers));
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}

// one block: the bucket of digit `digit` that holds the k_rem-th largest key; at the top digit K comes from
// C = the number of candidates (all that the histogram counted), Q and r: K = min(C, Q, max(ceil(C/2), ceil(Q/r)))
__global__ void __launch_bounds__(RT_AD_THREADS) k_budget_pick(int32_t* hist, int digit, long long Q, int r, BudgetSelect* sel) {
  const int b = 255 - threadIdx.x;  // thread order = buckets from the largest down
  const int h = hist[b];
  hist[b] = 0;  // zero for the next digit or the next pass
  long long k;
  if (digit == 3) {
    k = 0;  // (set below from the block total)
  } else {
    k = sel->k_rem;
    if (k == 0) return;
  }
  int total;
  const int above = block_exclusive_scan(h, &total);  // keys in larger buckets
  if (digit == 3) {
    const long long C = total;
    const long long half = (C + 1) / 2, share = (Q + r - 1) / r, wide = half > share ? half : share;
    k = C < Q ? C : Q;
    if (wide < k) k = wide;
    if (threadIdx.x == 0) {
      sel->C = (int)C;
      sel->K = (int)k;
      if (k == 0) { sel->prefix = 0xFFFFFFFFu; sel->k_rem = 0; }  // no key equals or exceeds it: no pixel is flagged
    }
    if (k == 0) return;
  }
  if (h > 0 && above < k && k <= above + h) {
    sel->prefix = (digit == 3 ? 0u : sel->prefix) | ((unsigned)b << (8 * digit));
    sel->k_rem = (int)(k - above);
  }
}

// keys of the tile's RT_AD_ITEMS-per-thread pixels, and how many of the thread's equal T
__device__ __forceinline__ int budget_tile_keys(const float* err_e, int n, float target, unsigned T, unsigned* key) {
  const int first = blockIdx.x * RT_AD_TILE + threadIdx.x * RT_AD_ITEMS;
  int ties = 0;
#pragma unroll
  for (int k = 0; k < RT_AD_ITEMS; ++k) {
    key[k] = first + k < n ? budget_key(err_e[first + k], target) : 0u;
    ties += key[k] == T;
  }
  return ties;
}

// per tile: the pixels whose key equals T
__global__ void __launch_bounds__(RT_AD_THREADS)
k_budget_ties(const float* err_e, int n, float target, const BudgetSelect* sel, int32_t* block_counts) {
  unsigned key[RT_AD_ITEMS];
  const int ties = budget_tile_keys(err_e, n, target, sel->prefix, key);
  int total;
  block_exclusive_scan(ties, &total);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// flags key > T, and key == T for the ties ranked below k_rem in pixel order (block_counts in: the tiles' tie
// offsets; out: the tiles' flag counts, as k_adaptive_combine leaves them)
__global__ void __launch_bounds__(RT_AD_THREADS)
k_budget_flags(const float* err_e, int n, float target, const BudgetSelect* sel, uint8_t* flags, int32_t* block_counts) {
  const unsigned T = sel->prefix;
  const int take = sel->k_rem;
  const int tile_ties = block_counts[blockIdx.x];
  unsigned key[RT_AD_ITEMS];
  const int ties = budget_tile_keys(err_e, n, target, T, key);
  int total;
  int rank = tile_ties + block_exclusive_scan(ties, &total);
  const int first = blockIdx.x * RT_AD_TILE + threadIdx.x * RT_AD_ITEMS;
  int count = 0;
#pragma unroll
  for (int k = 0; k < RT_AD_ITEMS; ++k) {
    bool f = key[k] > T;
    if (key[k] == T) f = rank++ < take;
    if (first + k < n) flags[first + k] = f ? 1 : 0;
    count += f;
  }
  block_exclusive_scan(count, &total);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

cudaError_t launch_adaptive_combine_budget(const ErrArgs& e, int pass, float floor_, float* sum_m, float* sum_v, int32_t* n_pass,
                                           float* err_e, int n_pixels, cudaStream_t st, LaunchInfo* info) {
  const int n = e.pix_list ? (int)e.n_list : n_pixels;
  if (n == 0) return cudaSuccess;
  k_adaptive_combine_budget<<<(n + RT_AD_THREADS - 1) / RT_AD_THREADS, RT_AD_THREADS, 0, st>>>(e.pix_list, n, e.err_mean, e.err_var, pass,
                                                                                                floor_, sum_m, sum_v, n_pass, err_e);
  if (info) info->n_launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_adaptive_select_budget(const float* err_e, int n_pixels, float target, long long Q, int r, BudgetSelect* sel,
                                          int32_t* hist, uint8_t* flags, int32_t* block_counts, int32_t* d_count, int32_t* next_list,
                                          int sm_count, cudaStream_t st, LaunchInfo* info) {
  const int nb = (n_pixels + RT_AD_TILE - 1) / RT_AD_TILE;
  if (nb == 0) return cudaMemsetAsync(d_count, 0, sizeof(int32_t), st);
  const int hb = std::min((n_pixels + RT_AD_THREADS - 1) / RT_AD_THREADS, std::max(sm_count, 1) * 8);
  for (int digit = 3; digit >= 0; --digit) {
    k_budget_hist<<<hb, RT_AD_THREADS, 0, st>>>(err_e, n_pixels, target, digit, sel, hist);
    k_budget_pick<<<1, RT_AD_THREADS, 0, st>>>(hist, digit, Q, r, sel);
  }
  k_budget_ties<<<nb, RT_AD_THREADS, 0, st>>>(err_e, n_pixels, target, sel, block_counts);
  k_adaptive_offsets<<<1, RT_AD_THREADS, 0, st>>>(block_counts, nb, &sel->scratch);
  k_budget_flags<<<nb, RT_AD_THREADS, 0, st>>>(err_e, n_pixels, target, sel, flags, block_counts);
  k_adaptive_offsets<<<1, RT_AD_THREADS, 0, st>>>(block_counts, nb, d_count);
  k_adaptive_scatter<<<nb, RT_AD_THREADS, 0, st>>>(nullptr, n_pixels, flags, block_counts, next_list);
  if (info) info->n_launches += 13;
  return cudaGetLastError();
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
