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
#include <cfloat>

#include "rt_launch.h"

#define RT_AD_THREADS 256
#define RT_AD_ITEMS 8                              // consecutive list entries per thread
#define RT_AD_TILE (RT_AD_THREADS * RT_AD_ITEMS)

// exclusive block-wide scan of one value per thread (RT_AD_THREADS threads); returns the block total in *total
template <typename T> __device__ T block_exclusive_scan(T v, T* total) {
  __shared__ T warp_sums[RT_AD_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  if (lane == 31) warp_sums[warp] = x;
  __syncthreads();
  T before = 0, all = 0;
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

// ---- budget modes (rt_render_adaptive_budget, rt_render_adaptive_rays): the next pass traces the longest prefix of the
// order (key descending, pixel index ascending) over the candidates (key > 0) whose weight fits the pass's target T
//   combine   as above, and per listed pixel (a pixel keeps what it has until traced again):
//               samples  err_e[px] = e; key = e > target ? bits(e) : 0, weight 1
//               rays     n_rays[px] += the pass's rays, weight[px] = w = ceil(n_rays / P), err_e[px] = the key as a float
//                        (e > target ? max(e / sqrt((P + 1) w), FLT_MIN) : 0); the selection then takes target 0
//   select    W = the candidates' weight and T from W, the budget left and r on the device; a radix select over four
//             8-bit digits finds the key at which the prefix is cut (64-bit weight histograms; one block per digit picks
//             the bucket where the weight from the top passes what is left); then every pixel with a larger key is
//             flagged, and the pixels with that key in index order while their inclusive weight stays within what is
//             left (ordered: per-tile weights, one ordered scan), and compacted like the threshold mode's flags
// sum_m, sum_v and n_pass of list entry i (pixel px) after the pass; the new sums in sm, sv; returns P
__device__ __forceinline__ int combine_entry(int i, int px, const float* em, const float* ev, int pass, float* sum_m, float* sum_v,
                                             int32_t* n_pass, float* sm, float* sv) {
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
  return P;
}

__global__ void __launch_bounds__(RT_AD_THREADS)
k_adaptive_combine_budget(const int32_t* list, int n, const float* em, const float* ev, int pass, float floor_, float* sum_m,
                          float* sum_v, int32_t* n_pass, float* err_e) {
  const int i = blockIdx.x * RT_AD_THREADS + threadIdx.x;
  if (i >= n) return;
  const int px = list ? list[i] : i;
  float sm[3], sv[3];
  const int P = combine_entry(i, px, em, ev, pass, sum_m, sum_v, n_pass, sm, sv);
  err_e[px] = adaptive_rel_error(sm, sv, P, floor_);
}

__global__ void __launch_bounds__(RT_AD_THREADS)
k_adaptive_combine_rays(const int32_t* list, int n, const float* em, const float* ev, const int32_t* rays, int pass, float target,
                        float floor_, float* sum_m, float* sum_v, int32_t* n_pass, long long* n_rays, int32_t* weight, float* err_e) {
  const int i = blockIdx.x * RT_AD_THREADS + threadIdx.x;
  if (i >= n) return;
  const int px = list ? list[i] : i;
  float sm[3], sv[3];
  const int P = combine_entry(i, px, em, ev, pass, sum_m, sum_v, n_pass, sm, sv);
  const long long nr = (pass == 0 ? 0ll : n_rays[px]) + rays[i];
  n_rays[px] = nr;
  const long long w = (nr + P - 1) / P;  // <= the most rays one pass of the pixel cost: fits an int32
  weight[px] = (int32_t)w;
  const float e = adaptive_rel_error(sm, sv, P, floor_);
  // e^2 / ((P + 1) w): the drop in relative variance one more pass buys, per predicted ray; FLT_MIN (normal, so no
  // flush to zero drops it) keeps every candidate's key above 0
  err_e[px] = e > target ? fmaxf(__fdiv_rn(e, __fsqrt_rn(__fmul_rn((float)(P + 1), (float)w))), FLT_MIN) : 0.f;
}

__device__ __forceinline__ unsigned budget_key(float e, float target) { return e > target ? __float_as_uint(e) : 0u; }

// weighted histogram of digit `digit` (bits 8 digit .. 8 digit + 7) of the candidate keys whose higher digits equal the
// prefix picked so far; lanes with the same bin are aggregated before the shared atomic
__global__ void __launch_bounds__(RT_AD_THREADS)
k_budget_hist(const float* err_e, const int32_t* weight, int n, float target, int digit, const BudgetSelect* sel,
              unsigned long long* hist) {
  __shared__ unsigned long long h[256];
  if (digit < 3 && sel->rem < 0) return;  // the top digit decided: no cut to find
  const unsigned hi_mask = digit == 3 ? 0u : 0xFFFFFFFFu << (8 * (digit + 1));
  const unsigned want = sel->prefix & hi_mask;
  const int lane = threadIdx.x & 31;
  h[threadIdx.x] = 0;
  __syncthreads();
  for (int base = blockIdx.x * RT_AD_THREADS; base < n; base += gridDim.x * RT_AD_THREADS) {
    const int i = base + threadIdx.x;
    int bin = -1;
    unsigned w = 0;
    if (i < n) {
      const unsigned key = budget_key(err_e[i], target);
      if (key && (key & hi_mask) == want) {
        bin = (key >> (8 * digit)) & 255;
        w = weight ? (unsigned)weight[i] : 1u;
      }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    unsigned long long sum = __popc(peers);
    if (weight) {  // (a kernel parameter: warp-uniform)
      sum = 0;
      for (int l = 0; l < 32; ++l) {
        const unsigned wl = __shfl_sync(0xffffffffu, w, l);
        if ((peers >> l) & 1u) sum += wl;
      }
    }
    if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&h[bin], sum);
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}

// one block: the bucket of digit `digit` in which the prefix is cut, the one where the weight from the top first exceeds
// rem; at the top digit the pass's target T = min(left, max(ceil(W/2), ceil(left/r))), W = the candidates' weight (all
// that the histogram counted), left = budget - *spent (without spent: budget); T = 0 or W <= T needs no cut
__global__ void __launch_bounds__(RT_AD_THREADS)
k_budget_pick(unsigned long long* hist, int digit, long long budget, const unsigned long long* spent, int r, BudgetSelect* sel) {
  const int b = 255 - threadIdx.x;  // thread order = buckets from the largest down
  const long long h = (long long)hist[b];
  hist[b] = 0;  // zero for the next digit or the next pass
  long long rem = 0;
  if (digit < 3) {
    rem = sel->rem;
    if (rem < 0) return;
  }
  long long total;
  const long long above = block_exclusive_scan(h, &total);  // weight in larger buckets
  if (digit == 3) {
    const long long W = total, left = spent ? budget - (long long)*spent : budget;
    long long T = 0;
    if (left > 0) {
      const long long half = (W + 1) / 2, share = (left + r - 1) / r;
      T = left < (half > share ? half : share) ? left : (half > share ? half : share);
    }
    if (threadIdx.x == 0) {
      sel->W = W;
      sel->want = T;
      // T = 0: no key equals or exceeds the cut, no pixel is flagged; W <= T: every key exceeds it, every candidate is
      if (T == 0 || W <= T) { sel->prefix = T == 0 ? 0xFFFFFFFFu : 0u; sel->rem = -1; }
    }
    if (T == 0 || W <= T) return;
    rem = T;
  }
  if (above <= rem && rem < above + h) {
    sel->prefix = (digit == 3 ? 0u : sel->prefix) | ((unsigned)b << (8 * digit));
    sel->rem = rem - above;
  }
}

// keys of the tile's RT_AD_ITEMS-per-thread pixels, and the weight of the thread's pixels whose key equals T
__device__ __forceinline__ unsigned long long budget_tile_keys(const float* err_e, const int32_t* weight, int n, float target, unsigned T,
                                                               unsigned* key) {
  const int first = blockIdx.x * RT_AD_TILE + threadIdx.x * RT_AD_ITEMS;
  unsigned long long ties = 0;
#pragma unroll
  for (int k = 0; k < RT_AD_ITEMS; ++k) {
    key[k] = first + k < n ? budget_key(err_e[first + k], target) : 0u;
    if (first + k < n && key[k] == T) ties += weight ? (unsigned)weight[first + k] : 1u;
  }
  return ties;
}

// per tile: the weight of the pixels whose key equals T
__global__ void __launch_bounds__(RT_AD_THREADS)
k_budget_ties(const float* err_e, const int32_t* weight, int n, float target, const BudgetSelect* sel, long long* tie_offsets) {
  unsigned key[RT_AD_ITEMS];
  const long long ties = (long long)budget_tile_keys(err_e, weight, n, target, sel->prefix, key);
  long long total;
  block_exclusive_scan(ties, &total);
  if (threadIdx.x == 0) tie_offsets[blockIdx.x] = total;
}

// one block: as k_adaptive_offsets, in 64 bits
__global__ void __launch_bounds__(RT_AD_THREADS) k_budget_tie_offsets(long long* tie_offsets, int nb, long long* sum) {
  long long carry = 0;
  for (int base = 0; base < nb; base += RT_AD_THREADS) {
    const int i = base + threadIdx.x;
    const long long v = i < nb ? tie_offsets[i] : 0;
    long long total;
    const long long ex = block_exclusive_scan(v, &total);
    if (i < nb) tie_offsets[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) *sum = carry;
}

// flags key > T, and key == T in pixel order while the ties' inclusive weight stays <= rem (tie_offsets: the tiles'
// exclusive tie weights; block_counts out: the tiles' flag counts, as k_adaptive_combine leaves them)
__global__ void __launch_bounds__(RT_AD_THREADS)
k_budget_flags(const float* err_e, const int32_t* weight, int n, float target, const BudgetSelect* sel, const long long* tie_offsets,
               uint8_t* flags, int32_t* block_counts) {
  const unsigned T = sel->prefix;
  const long long take = sel->rem;
  unsigned key[RT_AD_ITEMS];
  const long long ties = (long long)budget_tile_keys(err_e, weight, n, target, T, key);
  long long total;
  long long incl = tie_offsets[blockIdx.x] + block_exclusive_scan(ties, &total);
  const int first = blockIdx.x * RT_AD_TILE + threadIdx.x * RT_AD_ITEMS;
  int count = 0;
#pragma unroll
  for (int k = 0; k < RT_AD_ITEMS; ++k) {
    bool f = key[k] > T;
    if (first + k < n && key[k] == T) {
      incl += weight ? weight[first + k] : 1;
      f = incl <= take;
    }
    if (first + k < n) flags[first + k] = f ? 1 : 0;
    count += f;
  }
  int n_flags;
  block_exclusive_scan(count, &n_flags);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = n_flags;
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

cudaError_t launch_adaptive_combine_rays(const ErrArgs& e, int pass, float target, float floor_, float* sum_m, float* sum_v, int32_t* n_pass,
                                         long long* n_rays, int32_t* weight, float* err_e, int n_pixels, cudaStream_t st, LaunchInfo* info) {
  const int n = e.pix_list ? (int)e.n_list : n_pixels;
  if (n == 0) return cudaSuccess;
  k_adaptive_combine_rays<<<(n + RT_AD_THREADS - 1) / RT_AD_THREADS, RT_AD_THREADS, 0, st>>>(
      e.pix_list, n, e.err_mean, e.err_var, e.err_rays, pass, target, floor_, sum_m, sum_v, n_pass, n_rays, weight, err_e);
  if (info) info->n_launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_adaptive_select_budget(const float* err_e, const int32_t* weight, int n_pixels, float target, long long budget,
                                          const unsigned long long* spent, int r, BudgetSelect* sel, unsigned long long* hist, uint8_t* flags,
                                          int32_t* block_counts, long long* tie_offsets, int32_t* d_count, int32_t* next_list, int sm_count,
                                          cudaStream_t st, LaunchInfo* info) {
  const int nb = (n_pixels + RT_AD_TILE - 1) / RT_AD_TILE;
  if (nb == 0) return cudaMemsetAsync(d_count, 0, sizeof(int32_t), st);
  const int hb = std::min((n_pixels + RT_AD_THREADS - 1) / RT_AD_THREADS, std::max(sm_count, 1) * 8);
  for (int digit = 3; digit >= 0; --digit) {
    k_budget_hist<<<hb, RT_AD_THREADS, 0, st>>>(err_e, weight, n_pixels, target, digit, sel, hist);
    k_budget_pick<<<1, RT_AD_THREADS, 0, st>>>(hist, digit, budget, spent, r, sel);
  }
  k_budget_ties<<<nb, RT_AD_THREADS, 0, st>>>(err_e, weight, n_pixels, target, sel, tie_offsets);
  k_budget_tie_offsets<<<1, RT_AD_THREADS, 0, st>>>(tie_offsets, nb, &sel->scratch);
  k_budget_flags<<<nb, RT_AD_THREADS, 0, st>>>(err_e, weight, n_pixels, target, sel, tie_offsets, flags, block_counts);
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
