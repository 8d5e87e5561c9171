// rt_kernels.cuh — kernels templated on the arithmetic type; included by rt_kernels_f32.cu
// (float, multiply-add fusion on) and rt_kernels_f64.cu (double, --fmad=false).
//
//   k_resolve   OnOff / Flat / PointLight (render.py:52,65,157): one thread per pixel walks the
//               pixel's strata in the reference's order; shapes are staged through shared memory
//               in chunks by the whole block and read back as warp-wide broadcasts.
//   k_pt_mega   PathTracer (render.py:99-139) as a megakernel: one thread per pixel, the N-ary
//               recursion unrolled into a depth-first walk over an explicit level stack, random
//               numbers drawn in exactly the reference's order.
//   k_probe     one-item-per-thread / one-stream probes behind the known-answer entry points.
#pragma once
#include "rt_launch.h"
#include "rt_bvh.cuh"

#define RT_RESOLVE_THREADS 256
#ifndef RT_RESOLVE_BVH_MINB
#define RT_RESOLVE_BVH_MINB 3
#endif
#define RT_MEGA_THREADS 128
#define RT_SMEM_SHAPE_BYTES (48 * 1024)

template <typename T> RT_DEV V3<T> load3(const double* p) { return mk3<T>((T)p[0], (T)p[1], (T)p[2]); }

// ---------------------------------------------------------------- pixel ownership
struct PixelMap {
  long long n_pixels;  // pixels this rank traces
  int width, rank, count, rows_mode, compact;
  // where pixel p = (col, row) of this rank's share is stored: its place in the full-size image, or — row
  // partition with RT_ROWS_COMPACT — in the dense [owned rows][width] image of this rank
  RT_DEV long long at(long long p, int col, int row) const { return compact ? p : (long long)row * width + col; }
  RT_DEV void locate(long long p, int& col, int& row) const {
    int lrow;
    if (n_pixels < 0x7fffffffLL) {  // (uniform) a 64-bit division is ~100 instructions
      lrow = (int)((unsigned)p / (unsigned)width);
      col = (int)((unsigned)p - (unsigned)lrow * (unsigned)width);
    } else {
      lrow = (int)(p / width);
      col = (int)(p - (long long)lrow * width);
    }
    row = rows_mode ? rank + lrow * count : lrow;
  }
};

__host__ __device__ inline PixelMap make_pixel_map(const RenderArgs& a) {
  PixelMap pm;
  pm.width = a.width;
  pm.rows_mode = (a.part_mode == RT_PART_ROWS && a.part_count > 1);
  pm.rank = a.part_rank;
  pm.count = a.part_count;
  pm.compact = pm.rows_mode && a.rows_compact;
  int rows = a.height;
  if (pm.rows_mode) rows = (a.height - a.part_rank + a.part_count - 1) / a.part_count;
  if (rows < 0) rows = 0;
  pm.n_pixels = (long long)rows * a.width;
  return pm;
}

// List mode of the pixel map (the error-map kernels' sparse passes): with e.pix_list set, the tasks run over
// its n_list entries and entry p is the full-image pixel pix_list[p]; otherwise over the image
__host__ __device__ inline PixelMap make_pixel_map_list(const RenderArgs& a, const ErrArgs& e) {
  PixelMap pm = make_pixel_map(a);
  if (e.pix_list) pm.n_pixels = e.n_list;
  return pm;
}
RT_DEV void locate_listed(const PixelMap& pm, const ErrArgs& e, long long p, int& col, int& row) {
  if (e.pix_list) {
    const unsigned px = (unsigned)__ldg(e.pix_list + p);
    row = (int)(px / (unsigned)pm.width);
    col = (int)(px - (unsigned)row * (unsigned)pm.width);
  } else {
    pm.locate(p, col, row);
  }
}

RT_DEV bool stratum_is_mine(const RenderArgs& a, int s) {
  return !(a.part_mode == RT_PART_SPP && a.part_count > 1) || (s % a.part_count) == a.part_rank;
}

// row split with the exchange folded into the kernel: the pixel goes to every rank's image.  Out of line:
// the unrolled stores (24 per call site) would otherwise sit in the instruction stream of every render kernel
static __device__ __noinline__ void store_pixel_peers(float* const* peer_out, int n_peers, long long off, float r, float g, float b) {
#pragma unroll 1
  for (int k = 0; k < n_peers; ++k) {
    float* o = peer_out[k] + 3 * off;
    o[0] = r; o[1] = g; o[2] = b;
  }
}

template <typename T> RT_DEV void store_pixel(const RenderArgs& a, long long off, V3<T> c) {
  if (a.n_peers > 0) {
    store_pixel_peers(a.peer_out, a.n_peers, off, (float)c.x, (float)c.y, (float)c.z);
  } else if (a.out_f64) {
    double* o = (double*)a.out_rgb + 3 * off;
    o[0] = (double)c.x; o[1] = (double)c.y; o[2] = (double)c.z;
  } else {
    float* o = (float*)a.out_rgb + 3 * off;
    o[0] = (float)c.x; o[1] = (float)c.y; o[2] = (float)c.z;
  }
}

RT_DEV void block_count_add(unsigned long long* counter, unsigned int v) {
  v = __reduce_add_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(counter, (unsigned long long)v);
}

// cooperative copy global -> shared memory, 16 B per thread (both sides 16-byte aligned)
RT_DEV void stage_bytes(void* sh, const void* g, size_t bytes) {
  const uint4* src = reinterpret_cast<const uint4*>(g);
  uint4* dst = reinterpret_cast<uint4*>(sh);
  const int n16 = (int)(bytes / 16);
  for (int i = threadIdx.x; i < n16; i += blockDim.x) dst[i] = __ldg(src + i);
}
// shapes [c0, c1) of a [n][12] array
template <typename T> RT_DEV void stage_shapes(T* sh, const T* g, int c0, int c1) {
  stage_bytes(sh, g + 12 * (size_t)c0, (size_t)(c1 - c0) * 12 * sizeof(T));
}
#define RT_PLANES_SMEM_MAX 341  // plane records kept in shared memory next to the sphere chunk (16 KB)

// primary ray of sample (col,row,stratum) — fp64 generation, rounded to T
template <typename T>
RT_DEV Ray<T> primary_ray(const RenderArgs& a, int col, int row, int s, Pcg& aa) {
  double up = 0.5, vp = 0.5;
  if (a.S > 0) jitter_f64(aa, s % a.S, s / a.S, a.S, up, vp);
  V3<double> o, d;
  camera_ray_f64(a.cam, a.width, a.height, col, row, up, vp, o, d);
  Ray<T> r;
  r.o = cast3<T>(o);
  r.d = cast3<T>(d);
  r.tmin = (T)1.0e-5;
  r.tmax = Num<T>::inf();
  return r;
}

// ---------------------------------------------------------------- shading shared by kernels and probes
template <typename T> RT_DEV V3<T> flat_color(const SceneView<T>& sc, const Hit<T>& h) {  // render.py:70-74
  const DevMaterial& mat = sc.materials[sc.material[h.idx]];
  return pigment_color<T>(sc.pigments, mat.brdf_pigment, h.u, h.v) +
         pigment_color<T>(sc.pigments, mat.emitted_pigment, h.u, h.v);
}

// world.py:72-75: the segment from the hit point to the light
template <typename T> RT_DEV Ray<T> shadow_ray(V3<T> light_pos, V3<T> point) {
  Ray<T> r;
  r.o = point;
  r.d = light_pos - point;
  r.tmin = (T)1e-2 / Num<T>::sqrt(dot(r.d, r.d));
  r.tmax = (T)1;
  return r;
}

// render.py:172-191 for one visible light
template <typename T>
RT_DEV V3<T> light_term(const SceneView<T>& sc, const Hit<T>& h, V3<T> ray_dir, int l) {
  const DevLight& L = sc.lights[l];
  const DevMaterial& mat = sc.materials[sc.material[h.idx]];
  V3<T> lp = load3<T>(L.pos);
  V3<T> distance_vec = h.point - lp;
  T distance = Num<T>::sqrt(dot(distance_vec, distance_vec));
  V3<T> in_dir = ((T)1 / distance) * distance_vec;
  T cos_theta = Num<T>::max((T)0, normalized_dot(-in_dir, h.normal));
  T ratio = (T)L.radius / distance;
  T distance_factor = (L.radius > 0) ? ratio * ratio : (T)1;
  V3<T> b = brdf_eval<T>(sc, mat, h.normal, in_dir, -ray_dir, h.u, h.v);
  V3<T> lc = load3<T>(L.color);
  return mk3<T>(b.x * lc.x * cos_theta * distance_factor, b.y * lc.y * cos_theta * distance_factor,
                b.z * lc.z * cos_theta * distance_factor);
}

// ---------------------------------------------------------------- k_resolve
// `chunk` = shapes (fp64) or sphere PAIRS (fp32) staged per sweep step; everything in one chunk when
// it fits.  fp32 keeps the plane records in a small resident block and sweeps packed sphere pairs;
// crossed spheres are collected over all chunks and resolved once from global memory.
template <typename T, bool BVH>
__global__ void __launch_bounds__(RT_RESOLVE_THREADS, BVH ? RT_RESOLVE_BVH_MINB : 2)
k_resolve(const __grid_constant__ SceneView<T> sc, const __grid_constant__ RenderArgs a, const int chunk) {
  constexpr bool F32 = sizeof(T) == 4;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = sc.n_shapes, n_planes = sc.n_shapes - sc.n_spheres;
  const int n_units = F32 ? sc.n_pairs : n;
  const bool single = n_units <= chunk;
  // fp32 layout: [plane records (if few)][pair chunk]; fp64 layout: [shape chunk]
  const bool planes_smem = F32 && n_planes <= RT_PLANES_SMEM_MAX;
  const float* planes_g = F32 ? reinterpret_cast<const float*>(sc.packed) + 24 * (size_t)sc.n_pairs : nullptr;
  float* sh_planes = reinterpret_cast<float*>(smem_raw);
  float4* sh_pairs = reinterpret_cast<float4*>(smem_raw + (planes_smem ? (size_t)n_planes * 48 : 0));
  T* sh = reinterpret_cast<T*>(smem_raw);
  const float* planes = planes_smem ? sh_planes : planes_g;

  const PixelMap pm = make_pixel_map(a);
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = p < pm.n_pixels;
  int col = 0, row = 0;
  if (active) pm.locate(p, col, row);
  const long long pix = (long long)row * a.width + col;
  const int S2 = a.S > 0 ? a.S * a.S : 1;

  constexpr bool bvh = BVH;  // hierarchy traversal: nothing is staged, every thread walks the tree
  if (bvh) {
  } else if (F32) {
    if (planes_smem) stage_bytes(sh_planes, planes_g, (size_t)n_planes * 48);
    if (single) stage_bytes(sh_pairs, sc.packed, (size_t)sc.n_pairs * 96);
    __syncthreads();
  } else if (single) {
    stage_shapes(sh, sc.invm, 0, n);
    __syncthreads();
  }
  Pcg aa;
  aa.inc = a.aa_inc;
  aa.state = (a.S > 0 && active) ? pcg_jump(a.aa_state, 2ull * (unsigned long long)pix * S2, a.jump) : 0;

  V3<T> cum = mk3<T>((T)0, (T)0, (T)0);
  int last_hit = -1;
  unsigned int n_closest = 0, n_shadow = 0, n_samples = 0;
  const V3<T> background = load3<T>(a.background);

  for (int s = 0; s < S2; ++s) {  // block-uniform trip count
    const bool mine = active && stratum_is_mine(a, s);
    Ray<T> ray;
    if (active) ray = primary_ray<T>(a, col, row, s, aa);  // draws are consumed for every stratum
    // ---- closest hit: all threads of the block sweep the shape chunks together
    T best_t = Num<T>::inf();
    int best = -1;
    if (bvh) {
      if (mine) closest_bvh<T>(sc, ray, best_t, best);
    } else if constexpr (F32) {
      int cand[RT_CAND_CAP];
      int nc = 0;
      PackedRay pr;
      if (mine) pr = pack_ray(ray, sc.gate_a, sc.gate_t);
      if (single) {
        if (mine) sweep_pairs(sh_pairs, 0, 0, sc.n_pairs, pr, cand, nc);
      } else {
        for (int c0 = 0; c0 < sc.n_pairs; c0 += chunk) {
          const int c1 = min(c0 + chunk, sc.n_pairs);
          __syncthreads();
          stage_bytes(sh_pairs, sc.packed + 24 * (size_t)c0, (size_t)(c1 - c0) * 96);
          __syncthreads();
          if (mine) sweep_pairs(sh_pairs, c0, c0, c1, pr, cand, nc);
        }
      }
      if (mine) {
        resolve_candidates(sc.invm, sc.n_spheres, cand, nc, ray, best_t, best);
        scan_plane_block(planes, sc.n_spheres, n_planes, sc.orig, ray, best_t, best);
      }
    } else {
      if (single) {
        if (mine) scan_closest<T>(sh, 0, n, sc.n_spheres, sc.orig, ray, best_t, best);
      } else {
        for (int c0 = 0; c0 < n; c0 += chunk) {
          int c1 = min(c0 + chunk, n);
          __syncthreads();
          stage_shapes(sh, sc.invm, c0, c1);
          __syncthreads();
          if (mine) scan_closest<T>(sh, c0, c1, sc.n_spheres, sc.orig, ray, best_t, best);
        }
      }
    }
    if (mine) { ++n_closest; ++n_samples; }
    V3<T> color = background;
    Hit<T> h;
    h.idx = -1;
    if (mine && best >= 0) {
      finish_hit<T>(sc, ray, best_t, best, h);
      if (a.algorithm == RT_ALGO_ONOFF) color = load3<T>(a.onoff);
      else if (a.algorithm == RT_ALGO_FLAT) color = flat_color<T>(sc, h);
      else {  // render.py:163-167
        const DevMaterial& mat = sc.materials[sc.material[h.idx]];
        color = load3<T>(a.ambient) + pigment_color<T>(sc.pigments, mat.emitted_pigment, h.u, h.v);
      }
    }
    if (mine) last_hit = (best >= 0) ? sc.orig[best] : -1;
    if (a.algorithm == RT_ALGO_POINTLIGHT) {
      for (int l = 0; l < sc.n_lights; ++l) {  // render.py:168-191
        const bool need = mine && best >= 0;
        Ray<T> sr;
        if (need) { sr = shadow_ray<T>(load3<T>(sc.lights[l].pos), h.point); ++n_shadow; }
        bool blocked = false;
        if (bvh) {
          if (need) blocked = any_bvh<T>(sc, sr);
        } else if constexpr (F32) {
          int cand[RT_CAND_CAP];
          int nc = 0;
          PackedRay pr;
          if (need) { pr = pack_ray(sr, sc.gate_a, sc.gate_t); blocked = any_plane_blocks(planes, n_planes, sr); }
          if (single) {
            if (need && !blocked) sweep_pairs(sh_pairs, 0, 0, sc.n_pairs, pr, cand, nc);
          } else if (__syncthreads_or(need && !blocked)) {
            for (int c0 = 0; c0 < sc.n_pairs; c0 += chunk) {
              const int c1 = min(c0 + chunk, sc.n_pairs);
              __syncthreads();
              stage_bytes(sh_pairs, sc.packed + 24 * (size_t)c0, (size_t)(c1 - c0) * 96);
              __syncthreads();
              if (need && !blocked) sweep_pairs(sh_pairs, c0, c0, c1, pr, cand, nc);
            }
          }
          if (need && !blocked) blocked = any_candidate_blocks(sc.invm, sc.n_spheres, cand, nc, sr);
        } else {
          if (single) {
            if (need) blocked = scan_any<T>(sh, 0, n, sc.n_spheres, sr);
          } else if (__syncthreads_or(need)) {
            for (int c0 = 0; c0 < n; c0 += chunk) {
              int c1 = min(c0 + chunk, n);
              __syncthreads();
              stage_shapes(sh, sc.invm, c0, c1);
              __syncthreads();
              if (need && !blocked) blocked = scan_any<T>(sh, c0, c1, sc.n_spheres, sr);
            }
          }
        }
        if (need && !blocked) color = color + light_term<T>(sc, h, ray.d, l);
      }
    }
    if (mine) cum = (a.S > 0) ? cum + color : color;
  }
  if (active) {
    if (a.S > 0) cum = ((T)1 / (T)(S2)) * cum;  // imagetracer.py:99-101
    store_pixel<T>(a, pm.at(p, col, row), cum);
    if (a.out_hit) a.out_hit[pm.at(p, col, row)] = a.hit_mode == RT_HIT_RAY_COUNT ? (int)(n_closest + n_shadow) : last_hit;
  }
  block_count_add(a.counters + CNT_CLOSEST, n_closest);
  block_count_add(a.counters + CNT_SHADOW, n_shadow);
  block_count_add(a.counters + CNT_SAMPLES, n_samples);
}

template <typename T>
cudaError_t launch_resolve_generic(const SceneView<T>& sc, const RenderArgs& a, cudaStream_t st, LaunchInfo* info) {
  PixelMap pm = make_pixel_map(a);
  if (pm.n_pixels == 0) return cudaSuccess;
  constexpr bool F32 = sizeof(T) == 4;
  // everything in one chunk while it fits 96 KB of shared memory, else 48 KB chunks
  void (*kern)(const SceneView<T>, const RenderArgs, const int) = sc.accel ? k_resolve<T, true> : k_resolve<T, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * RT_SMEM_SHAPE_BYTES + 16 * 1024);
  if (e != cudaSuccess) return e;
  const int n_planes = sc.n_shapes - sc.n_spheres;
  const size_t unit = F32 ? 96 : 12 * sizeof(T);
  const int n_units = F32 ? sc.n_pairs : sc.n_shapes;
  const size_t planes_bytes = (F32 && n_planes <= RT_PLANES_SMEM_MAX) ? (size_t)n_planes * 48 : 0;
  int chunk = (size_t)n_units * unit <= 2 * RT_SMEM_SHAPE_BYTES ? (n_units > 0 ? n_units : 1) : (int)(RT_SMEM_SHAPE_BYTES / unit);
  size_t smem = sc.accel ? 16 : planes_bytes + (size_t)chunk * unit;
  long long blocks = (pm.n_pixels + RT_RESOLVE_THREADS - 1) / RT_RESOLVE_THREADS;
  kern<<<(unsigned)blocks, RT_RESOLVE_THREADS, smem, st>>>(sc, a, chunk);
  if (info) { info->n_launches += 1; info->variant = 0; }
  return cudaGetLastError();
}

// ---------------------------------------------------------------- PathTracer, depth-first
template <typename T> struct Level {
  V3<T> P, nd, w;  // hit point; normal (diffuse) or mirror direction (specular); throughput of a child
  int remaining, depth, kind, origin;  // origin: sorted index of the shape the children start on
};

template <typename T> struct PtCtx {
  const SceneView<T>* sc;
  ScanSrc<T> src;  // scan data of all shapes (shared or global memory)
  V3<T> background;
  int N, max_depth, rr_limit;
  unsigned int n_rays;
};

// BVH is a template parameter, not a run-time branch: with the walk inlined beside the linear scan the
// megakernel went from 96 to 128 registers and lost 12 % of its speed on the linear path
template <typename T, bool BVH = false>
RT_DEV bool trace_closest(const SceneView<T>& sc, const ScanSrc<T>& src, const Ray<T>& r, Hit<T>& h, int origin = -1) {
  T best_t = Num<T>::inf();
  int best = -1;
  if constexpr (BVH) closest_bvh<T>(sc, r, best_t, best, origin);
  else closest_all<T>(sc, src, r, best_t, best, origin);
  h.idx = -1;
  if (best < 0) return false;
  finish_hit<T>(sc, r, best_t, best, h);
  return true;
}

// PathTracer.__call__(ray) with ray.depth = depth0 (render.py:99-139).  The recursion becomes a
// walk over `stack`: a level is a surface interaction that still owes `remaining` scattered rays;
// the estimator is linear, so each traced ray adds throughput * (emitted | background) to the
// result.  Draw order = the reference's: roulette draw at the hit, then for each child its two
// scatter draws followed by everything its subtree draws.
template <typename T, int MAXL, bool BVH = false>
RT_DEV V3<T> pt_radiance(PtCtx<T>& cx, Ray<T> ray, int depth, Pcg& rng, int* primary_hit) {
  const SceneView<T>& sc = *cx.sc;
  Level<T> stack[MAXL];
  int top = -1;
  V3<T> acc = mk3<T>((T)0, (T)0, (T)0);
  V3<T> thr = mk3<T>((T)1, (T)1, (T)1);
  const T inv_n = (T)1 / (T)cx.N;
  bool first = true;
  int origin = -1;
  if (depth > cx.max_depth) return acc;  // render.py:100-101
  while (true) {
    Hit<T> h;
    bool found = trace_closest<T, BVH>(sc, cx.src, ray, h, origin);
    ++cx.n_rays;
    if (first) { if (primary_hit) *primary_hit = found ? sc.orig[h.idx] : -1; first = false; }
    if (!found) {
      acc = acc + mul3(thr, cx.background);
    } else {
      const DevMaterial& mat = sc.materials[sc.material[h.idx]];
      V3<T> hit_color = pigment_color<T>(sc.pigments, mat.brdf_pigment, h.u, h.v);
      V3<T> emitted = pigment_color<T>(sc.pigments, mat.emitted_pigment, h.u, h.v);
      acc = acc + mul3(thr, emitted);
      T lum = max3(hit_color);
      bool go_on = true;
      if (depth >= cx.rr_limit) {  // render.py:116-123
        T q = Num<T>::max((T)0.05, (T)1 - lum);
        if (pcg_random_float<T>(rng) > q) hit_color = ((T)1 / ((T)1 - q)) * hit_color;
        else go_on = false;
      }
      if (go_on && lum > (T)0) {
        if (depth < cx.max_depth) {
          Level<T>& L = stack[++top];
          L.P = h.point;
          L.kind = mat.brdf_kind;
          L.nd = (mat.brdf_kind == RT_BRDF_DIFFUSE) ? h.normal : specular_dir<T>(ray.d, h.normal);
          L.w = inv_n * mul3(thr, hit_color);
          L.remaining = cx.N;
          L.depth = depth + 1;
          L.origin = h.idx;
        } else if (mat.brdf_kind == RT_BRDF_DIFFUSE) {
          // the reference still scatters N rays here and cuts them at depth > max_depth
          pcg_skip(rng, 2u * (unsigned)cx.N);
        }
      }
    }
    if (top < 0) break;
    Level<T>& L = stack[top];
    ray.o = L.P;
    ray.tmax = Num<T>::inf();
    if (L.kind == RT_BRDF_DIFFUSE) {
      T u1 = pcg_random_float<T>(rng);
      T u2 = pcg_random_float<T>(rng);
      ray.d = diffuse_dir<T>(L.nd, u1, u2);
      ray.tmin = (T)1.0e-3;
    } else {
      ray.d = L.nd;
      ray.tmin = (T)1e-5;
    }
    thr = L.w;
    depth = L.depth;
    origin = L.origin;
    if (--L.remaining == 0) --top;  // the slot is free for the child's own level
  }
  return acc;
}

template <typename T, int MAXL, bool BVH>
__global__ void __launch_bounds__(RT_MEGA_THREADS)
k_pt_mega(const __grid_constant__ SceneView<T> sc, const __grid_constant__ RenderArgs a, const int in_smem) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ScanSrc<T> src = global_src<T>(sc);
  if (in_smem) {
    if constexpr (sizeof(T) == 4) {
      const size_t bytes = (size_t)sc.n_pairs * 96 + (size_t)(sc.n_shapes - sc.n_spheres) * 48;
      stage_bytes(smem_raw, sc.packed, bytes);
      src.pairs = reinterpret_cast<const float4*>(smem_raw);
      src.planes = reinterpret_cast<const float*>(smem_raw) + 24 * (size_t)sc.n_pairs;
    } else {
      T* sh = reinterpret_cast<T*>(smem_raw);
      stage_shapes(sh, sc.invm, 0, sc.n_shapes);
      src.xf = sh;
    }
    __syncthreads();
  }
  const PixelMap pm = make_pixel_map(a);
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned int n_samples = 0;
  PtCtx<T> cx;
  cx.sc = &sc; cx.src = src; cx.background = load3<T>(a.background);
  cx.N = a.num_of_rays; cx.max_depth = a.max_depth; cx.rr_limit = a.rr_limit; cx.n_rays = 0;
  if (p < pm.n_pixels) {
    int col, row;
    pm.locate(p, col, row);
    const long long pix = (long long)row * a.width + col;
    const int S2 = a.S > 0 ? a.S * a.S : 1;
    Pcg aa;
    aa.inc = a.aa_inc;
    aa.state = (a.S > 0) ? pcg_jump(a.aa_state, 2ull * (unsigned long long)pix * S2, a.jump) : 0;
    // the pixel's sum over its strata is kept in fp64 whatever T is: a sequential fp32 sum of 1 024 equal
    // samples (a sky pixel at 1 024 spp) is off by 3e-5, and it costs three additions per SAMPLE
    V3<double> cum = mk3<double>(0.0, 0.0, 0.0);
    int last_hit = -1;
    for (int s = 0; s < S2; ++s) {
      Ray<T> ray = primary_ray<T>(a, col, row, s, aa);
      if (!stratum_is_mine(a, s)) continue;
      const unsigned long long k = (unsigned long long)pix * S2 + s;
      Pcg rng;
      if (a.rng_mode == RT_RNG_REPLAY) { rng.state = a.replay[k]; rng.inc = a.pt_inc; }
      else rng = pcg_seed(a.pt_state, (a.pt_inc >> 1) + k);
      const V3<double> c = cast3<double>(pt_radiance<T, MAXL, BVH>(cx, ray, 0, rng, &last_hit));
      cum = (a.S > 0) ? mk3<double>(__dadd_rn(cum.x, c.x), __dadd_rn(cum.y, c.y), __dadd_rn(cum.z, c.z)) : c;
      ++n_samples;
    }
    if (a.S > 0) {  // imagetracer.py:99-101
      const double inv = __ddiv_rn(1.0, (double)S2);
      cum = mk3<double>(__dmul_rn(inv, cum.x), __dmul_rn(inv, cum.y), __dmul_rn(inv, cum.z));
    }
    store_pixel<double>(a, pm.at(p, col, row), cum);
    if (a.out_hit) a.out_hit[pm.at(p, col, row)] = a.hit_mode == RT_HIT_RAY_COUNT ? (int)cx.n_rays : last_hit;
  }
  block_count_add(a.counters + CNT_CLOSEST, cx.n_rays);
  block_count_add(a.counters + CNT_SAMPLES, n_samples);
}

template <typename T>
cudaError_t launch_pt_mega(const SceneView<T>& sc, const RenderArgs& a, cudaStream_t st, LaunchInfo* info) {
  PixelMap pm = make_pixel_map(a);
  if (pm.n_pixels == 0) return cudaSuccess;
  size_t bytes = sizeof(T) == 4 ? (size_t)sc.n_pairs * 96 + (size_t)(sc.n_shapes - sc.n_spheres) * 48
                                : (size_t)sc.n_shapes * 12 * sizeof(T);
  int in_smem = bytes <= RT_SMEM_SHAPE_BYTES;
  size_t smem = in_smem ? (bytes ? bytes : 16) : 16;
  long long blocks = (pm.n_pixels + RT_MEGA_THREADS - 1) / RT_MEGA_THREADS;
  int need = a.num_of_rays == 1 ? 1 : a.max_depth;
  if (sc.accel) {  // the hierarchy walk reads global memory: nothing is staged
    in_smem = 0;
    smem = 16;
    if (need <= 4) k_pt_mega<T, 4, true><<<(unsigned)blocks, RT_MEGA_THREADS, smem, st>>>(sc, a, in_smem);
    else if (need <= 16) k_pt_mega<T, 16, true><<<(unsigned)blocks, RT_MEGA_THREADS, smem, st>>>(sc, a, in_smem);
    else if (need <= 64) k_pt_mega<T, 64, true><<<(unsigned)blocks, RT_MEGA_THREADS, smem, st>>>(sc, a, in_smem);
    else return cudaErrorInvalidValue;
  } else if (need <= 4) k_pt_mega<T, 4, false><<<(unsigned)blocks, RT_MEGA_THREADS, smem, st>>>(sc, a, in_smem);
  else if (need <= 16) k_pt_mega<T, 16, false><<<(unsigned)blocks, RT_MEGA_THREADS, smem, st>>>(sc, a, in_smem);
  else if (need <= 64) k_pt_mega<T, 64, false><<<(unsigned)blocks, RT_MEGA_THREADS, smem, st>>>(sc, a, in_smem);
  else return cudaErrorInvalidValue;
  if (info) { info->n_launches += 1; info->variant = RT_VARIANT_MEGA; }
  return cudaGetLastError();
}

// ---------------------------------------------------------------- probes
template <typename T> RT_DEV Ray<T> ray_from8(const double* q) {
  Ray<T> r;
  r.o = mk3<T>((T)q[0], (T)q[1], (T)q[2]);
  r.d = mk3<T>((T)q[3], (T)q[4], (T)q[5]);
  r.tmin = (T)q[6];
  r.tmax = (T)q[7];
  return r;
}
template <typename T> RT_DEV void ray_to8(const Ray<T>& r, double* q) {
  q[0] = r.o.x; q[1] = r.o.y; q[2] = r.o.z; q[3] = r.d.x; q[4] = r.d.y; q[5] = r.d.z;
  q[6] = r.tmin; q[7] = r.tmax;
}

// Renderer.__call__(ray) for one explicit ray (render.py:52,65,99,157), shapes read from global memory
template <typename T>
RT_DEV V3<T> renderer_call(const SceneView<T>& sc, const RenderArgs& a, const Ray<T>& ray, int depth, Pcg& rng,
                           unsigned long long* n_closest, unsigned long long* n_shadow) {
  if (a.algorithm == RT_ALGO_PATHTRACING) {
    PtCtx<T> cx;
    cx.sc = &sc; cx.src = global_src<T>(sc); cx.background = load3<T>(a.background);
    cx.N = a.num_of_rays; cx.max_depth = a.max_depth; cx.rr_limit = a.rr_limit; cx.n_rays = 0;
    V3<T> c = (a.num_of_rays == 1) ? pt_radiance<T, 1>(cx, ray, depth, rng, nullptr)
                                   : pt_radiance<T, 64>(cx, ray, depth, rng, nullptr);
    *n_closest += cx.n_rays;
    return c;
  }
  Hit<T> h;
  *n_closest += 1;
  const ScanSrc<T> src = global_src<T>(sc);
  if (!trace_closest<T>(sc, src, ray, h)) return load3<T>(a.background);
  if (a.algorithm == RT_ALGO_ONOFF) return load3<T>(a.onoff);
  if (a.algorithm == RT_ALGO_FLAT) return flat_color<T>(sc, h);
  const DevMaterial& mat = sc.materials[sc.material[h.idx]];
  V3<T> color = load3<T>(a.ambient) + pigment_color<T>(sc.pigments, mat.emitted_pigment, h.u, h.v);
  for (int l = 0; l < sc.n_lights; ++l) {
    Ray<T> sr = shadow_ray<T>(load3<T>(sc.lights[l].pos), h.point);
    *n_shadow += 1;
    if (!any_all<T>(sc, src, sr)) color = color + light_term<T>(sc, h, ray.d, l);
  }
  return color;
}

template <typename T>
__global__ void k_probe(const __grid_constant__ SceneView<T> sc, const __grid_constant__ RenderArgs a, const ProbeArgs p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  switch (p.what) {
    case PROBE_TRACE: {  // one thread, one PCG stream, rays in order
      if (i != 0) return;
      Pcg rng;
      rng.state = p.pcg[0]; rng.inc = p.pcg[1];
      unsigned long long nc = 0, ns = 0;
      for (int k = 0; k < p.n; ++k) {
        Ray<T> r = ray_from8<T>(p.in + 8 * (size_t)k);
        V3<T> c = renderer_call<T>(sc, a, r, p.depth ? p.depth[k] : 0, rng, &nc, &ns);
        p.out[3 * k] = c.x; p.out[3 * k + 1] = c.y; p.out[3 * k + 2] = c.z;
      }
      p.pcg[0] = rng.state;
      atomicAdd(a.counters + CNT_CLOSEST, nc);
      atomicAdd(a.counters + CNT_SHADOW, ns);
      atomicAdd(a.counters + CNT_SAMPLES, (unsigned long long)p.n);
      return;
    }
    case PROBE_INTERSECT: {
      if (i >= p.n) return;
      Ray<T> r = ray_from8<T>(p.in + 8 * (size_t)i);
      Hit<T> h;
      rt_hit out;
      memset(&out, 0, sizeof(out));
      T best_t = Num<T>::inf();
      int best = -1;
      closest_all<T>(sc, global_src<T>(sc), r, best_t, best);
      if (best < 0) { out.shape = -1; out.material = -1; }
      else {
        finish_hit<T>(sc, r, best_t, best, h, p.aux != 0, true);
        out.shape = sc.orig[best]; out.material = sc.material[best]; out.t = h.t;
        out.world_point[0] = h.point.x; out.world_point[1] = h.point.y; out.world_point[2] = h.point.z;
        out.normal[0] = h.normal.x; out.normal[1] = h.normal.y; out.normal[2] = h.normal.z;
        out.uv[0] = h.u; out.uv[1] = h.v;
      }
      p.hits[i] = out;
      return;
    }
    case PROBE_VISIBLE: {
      if (i >= p.n) return;
      const double* q = p.in + 6 * (size_t)i;
      Ray<T> sr = shadow_ray<T>(mk3<T>((T)q[0], (T)q[1], (T)q[2]), mk3<T>((T)q[3], (T)q[4], (T)q[5]));
      p.flags[i] = any_all<T>(sc, global_src<T>(sc), sr) ? 0 : 1;
      return;
    }
    case PROBE_PIGMENT: {
      if (i >= p.n) return;
      V3<T> c = pigment_color<T>(sc.pigments, p.aux, (T)p.in[2 * i], (T)p.in[2 * i + 1]);
      p.out[3 * i] = c.x; p.out[3 * i + 1] = c.y; p.out[3 * i + 2] = c.z;
      return;
    }
    case PROBE_SCATTER: {  // sequential: one stream
      if (i != 0) return;
      Pcg rng;
      rng.state = p.pcg[0]; rng.inc = p.pcg[1];
      const DevMaterial& mat = sc.materials[p.aux];
      for (int k = 0; k < p.n; ++k) {
        const double* q = p.in + 9 * (size_t)k;
        V3<T> in_dir = mk3<T>((T)q[0], (T)q[1], (T)q[2]);
        V3<T> nrm = mk3<T>((T)q[6], (T)q[7], (T)q[8]);
        Ray<T> r;
        r.o = mk3<T>((T)q[3], (T)q[4], (T)q[5]);
        r.tmax = Num<T>::inf();
        if (mat.brdf_kind == RT_BRDF_DIFFUSE) {
          T u1 = pcg_random_float<T>(rng);
          T u2 = pcg_random_float<T>(rng);
          r.d = diffuse_dir<T>(nrm, u1, u2);
          r.tmin = (T)1.0e-3;
        } else {
          r.d = specular_dir<T>(in_dir, nrm);
          r.tmin = (T)1e-5;
        }
        ray_to8<T>(r, p.out + 8 * (size_t)k);
      }
      p.pcg[0] = rng.state;
      return;
    }
    case PROBE_ONB: {
      if (i >= p.n) return;
      V3<T> nrm = mk3<T>((T)p.in[3 * i], (T)p.in[3 * i + 1], (T)p.in[3 * i + 2]);
      V3<T> e1, e2;
      onb_from_z<T>(nrm, e1, e2);
      double* o = p.out + 9 * (size_t)i;
      o[0] = e1.x; o[1] = e1.y; o[2] = e1.z; o[3] = e2.x; o[4] = e2.y; o[5] = e2.z;
      o[6] = nrm.x; o[7] = nrm.y; o[8] = nrm.z;
      return;
    }
    case PROBE_PCG_DRAW: {
      if (i != 0) return;
      Pcg rng;
      rng.state = p.pcg[0]; rng.inc = p.pcg[1];
      for (int k = 0; k < p.n; ++k) p.draws[k] = pcg_random(rng);
      p.pcg[0] = rng.state;
      return;
    }
    case PROBE_PCG_SEED: {
      if (i != 0) return;
      Pcg rng = pcg_seed(p.pcg[0], p.pcg[1]);
      p.pcg[0] = rng.state; p.pcg[1] = rng.inc;
      return;
    }
    case PROBE_CAMERA_RAYS: {  // every sample of the image, jitter by jump-ahead
      const int S2 = a.S > 0 ? a.S * a.S : 1;
      const long long total = (long long)a.width * a.height * S2;
      if (i >= total) return;
      const long long pix = i / S2;
      const int s = (int)(i - pix * S2);
      Pcg aa;
      aa.inc = a.aa_inc;
      aa.state = (a.S > 0) ? pcg_jump(a.aa_state, 2ull * (unsigned long long)i, a.jump) : 0;
      Ray<T> r = primary_ray<T>(a, (int)(pix % a.width), (int)(pix / a.width), s, aa);
      ray_to8<T>(r, p.out + 8 * (size_t)i);
      return;
    }
    case PROBE_CAMERA_UV: {  // Camera.fire_ray(u, v)
      if (i >= p.n) return;
      V3<double> o, d;
      camera_fire_f64(a.cam, p.in[2 * i], p.in[2 * i + 1], o, d);
      Ray<T> r;
      r.o = cast3<T>(o); r.d = cast3<T>(d); r.tmin = (T)1.0e-5; r.tmax = Num<T>::inf();
      ray_to8<T>(r, p.out + 8 * (size_t)i);
      return;
    }
  }
}

template <typename T>
cudaError_t launch_probe(const SceneView<T>& sc, const RenderArgs& a, const ProbeArgs& p, cudaStream_t st) {
  long long n = p.n;
  if (p.what == PROBE_CAMERA_RAYS) n = (long long)a.width * a.height * (a.S > 0 ? a.S * a.S : 1);
  if (p.what == PROBE_TRACE || p.what == PROBE_SCATTER || p.what == PROBE_PCG_DRAW || p.what == PROBE_PCG_SEED) n = 1;
  if (n <= 0) return cudaSuccess;
  unsigned blocks = (unsigned)((n + 127) / 128);
  // the single-stream probes walk a 64-level stack in local memory
  k_probe<T><<<blocks, 128, 0, st>>>(sc, a, p);
  return cudaGetLastError();
}
