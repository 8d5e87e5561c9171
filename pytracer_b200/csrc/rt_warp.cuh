// rt_warp.cuh — PathTracer (render.py:99-139) as a warp-cooperative wavefront (fp32).
//
// Why: on demo.txt 48 % of the samples trace one ray while 6.6 % trace up to 1 111; a thread-per-
// sample walk leaves most lanes idle.  Here a warp owns a group of pixels and keeps, in shared
// memory, a LIFO stack of *scatter records* — one per surface interaction that still owes
// num_of_rays scattered rays {point, normal | mirror direction, child throughput, depth, rng}.
// Every iteration the 32 lanes take the next 32 owed rays off the top of the stack (a record is
// shared by up to N consecutive lanes: broadcast reads), each lane scatters, traces and shades its
// ray, and the lanes whose ray must branch again push a new record; positions come from one ballot
// (warp-level compaction).  Lanes stay full whatever single samples do, and the closest-hit loop
// over the shapes stays perfectly convergent: all lanes walk the same shape list.
//
// The estimator is the reference's (N children per interaction, Russian roulette from rr_limit,
// children cut beyond max_depth); it is linear, so each traced ray adds
// throughput * (emitted | background) to its pixel.  Random numbers: a record carries a 64-bit
// state; child i owns z = mix64(state + (i+1)*phi64) (rt_pcg.cuh: child_stream) — its two scatter
// uniforms are the halves of z, a roulette draw is a PCG32 step from z — so the image depends only
// on (sample index, position in the tree) and not on lane assignment, GPU count or partition.
#pragma once
#include <type_traits>

#include "rt_kernels.cuh"

#define RT_WARP_MAX_THREADS 256
#ifndef RT_WARP_SPLIT
#define RT_WARP_SPLIT 1
#endif


struct __align__(16) ScatterRec {
  float4 a;  // P.xyz, meta (slot | kind << 5 | child depth << 6 (10 bits) | origin shape << 16 (0xFFFF: none))
  float4 b;  // nd.xyz (normal, or mirror direction for a specular surface), w.r
  float4 c;  // w.g, w.b, rng state lo, hi
};

struct WarpCfg {
  int cap;            // records per warp stack
  int group;          // pixels per task (G)
  int per_pixel;      // strata of a pixel traced by this rank (L)
  int rounds;         // ceil(G * L / 32)
  int per_warp_bytes;
  int shape_bytes;    // shared memory reserved for the shape block (0 = read from global)
  long long n_tasks;
  // values every iteration needs, precomputed so that they are constant-bank operands instead of
  // registers: background colour in fp32, 1/N, 1/spp, the multiply-shift magic for x / N
  float bg[3], inv_n, inv_spp;
  unsigned n_magic;
  double inv_w, inv_h, inv_s;  // 1 / width, 1 / height, 1 / samples_per_side (fp64, host-rounded)
  unsigned long long n_samples;  // samples this launch traces (all tasks), added to the counter once
};

// ---- error map (ERR instantiations) --------------------------------------------------------------------
// The L samples a pixel traces in one pass fall into B = min(L, 32 / G) batches: sample ls goes to batch
// ls mod (32 / G) and every ray of its tree inherits that batch through the 5-bit slot of its scatter record
// (slot = pixel in task * (32 / G) + batch).  The warp keeps the 32 batch sums [32][3] in shared memory;
// the squared standard error of the pass mean m follows from them when the task ends:
//   SE^2 = sum_b (T_b - n_b m)^2 / (n_b (B - 1) L)
// (unbiased for independent samples; B = L gives s^2 / L).
// RT_ERR_EST_PAIRED (S even) collapses pairs of strata instead: strata 2k and 2k + 1 (horizontal neighbours)
// land in batches 2j and 2j + 1 (bpp is even), so D_j = T_2j - T_2j+1 sums the pair differences of group j and
//   SE^2 = sum_j D_j^2 / L^2,   j < min(L, bpp) / 2
// (E[D_j^2] >= the pairs' variances: conservative under stratification, tight where radiance is smooth).
RT_DEV int err_batch_of(const ErrArgs& cfg, int ls) {
  return cfg.err_bpp == 32 ? (ls & 31) : ls - (int)(((unsigned)ls * cfg.err_magic) >> 16) * cfg.err_bpp;  // (ls < 32 when G > 1)
}
// Adds this lane's contribution to batch `slot` (all lanes call; `on`: the lane traced a ray).  Lanes of one
// record are contiguous and share the slot: a segmented scan over runs of equal slots, then one shared
// atomic per run, as ACC_SEG does for pixels.
RT_DEV void err_batch_add(float* bsum, int slot, bool on, V3<float> c, int lane) {
  const unsigned FULL = 0xffffffffu;
  if (__ballot_sync(FULL, on && (c.x != 0.f || c.y != 0.f || c.z != 0.f)) == 0u) return;
  const int key = on ? slot : 32 + lane;
  const int prev = __shfl_up_sync(FULL, key, 1);
  const unsigned heads = __ballot_sync(FULL, lane == 0 || prev != key);
  const int seg_start = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const float r = __shfl_up_sync(FULL, c.x, d);
    const float g = __shfl_up_sync(FULL, c.y, d);
    const float b = __shfl_up_sync(FULL, c.z, d);
    if (lane - d >= seg_start) { c.x += r; c.y += g; c.z += b; }
  }
  const bool tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
  if (on && tail && (c.x != 0.f || c.y != 0.f || c.z != 0.f)) {
    atomicAdd(&bsum[3 * slot + 0], c.x);
    atomicAdd(&bsum[3 * slot + 1], c.y);
    atomicAdd(&bsum[3 * slot + 2], c.z);
  }
}
// Pass mean m (the value the plain kernel stores, identical in all lanes) and SE^2 of pixel g of the task
// to list entry `entry`.  All lanes call.
RT_DEV void err_store(const ErrArgs& e, int L, const float* bsum, int g, long long entry, V3<float> m, int lane) {
  const unsigned FULL = 0xffffffffu;
  const int bpp = e.err_bpp, B = min(L, bpp);
  const bool paired = e.estimator == RT_ERR_EST_PAIRED;  // (a kernel parameter: warp-uniform)
  float tr = 0.f, tg = 0.f, tb = 0.f;
  if (paired) {
    if (lane < B / 2) {
      const float* t = bsum + 3 * (g * bpp + 2 * lane);
      const float dr = t[0] - t[3], dg = t[1] - t[4], db = t[2] - t[5];
      tr = __fmul_rn(dr, dr); tg = __fmul_rn(dg, dg); tb = __fmul_rn(db, db);  // (no fusion into the first add below)
    }
  } else if (lane < B) {
    const float n = (float)((L - 1 - lane) / bpp + 1);
    const float* t = bsum + 3 * (g * bpp + lane);
    const float dr = fmaf(-n, m.x, t[0]), dg = fmaf(-n, m.y, t[1]), db = fmaf(-n, m.z, t[2]);
    tr = dr * dr / n; tg = dg * dg / n; tb = db * db / n;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    tr += __shfl_xor_sync(FULL, tr, d);
    tg += __shfl_xor_sync(FULL, tg, d);
    tb += __shfl_xor_sync(FULL, tb, d);
  }
  if (lane == 0) {
    const float k = paired ? 1.f / ((float)L * (float)L) : 1.f / ((float)(B - 1) * (float)L);
    float* o = e.err_mean + 3 * entry;
    o[0] = m.x; o[1] = m.y; o[2] = m.z;
    float* v = e.err_var + 3 * entry;
    v[0] = tr * k; v[1] = tg * k; v[2] = tb * k;
  }
}

// SMALL instantiation: every table of the scene lives in shared memory at FIXED offsets (capacity for
// the largest small scene, 3.6 KB), re-packed by the staging loop into what the per-ray code reads:
//   SM_INVM / SM_M   [16][12] fp32 transforms, rows 0 and 1 interleaved column by column for the paired FP32
//                    pipe: {r0.x, r1.x, r0.y, r1.y}, {r0.z, r1.z, r0.w, r1.w}, then row 2 (three LDS.128 per shape)
//   SM_PLANE2        [8][8] row 2 of the inverse transforms of planes 2j and 2j + 1, interleaved:
//                    {x, x', y, y'}, {z, z', w, w'} (the odd plane of an odd count pairs with zeros)
//   SM_ORIG          [16] index in World.shapes
//   SM_SHAPE_MAT     [16] the shape's material as one int4 {brdf_kind, brdf_pigment, emitted_pigment, flags}
//                    (no material-index indirection)
//   SM_PIG           [32] 48-byte pigment records {kind, steps, tex_w, tex_h | c1.xyz, c2.x | c2.yz, texture handle}
//   SM_JUMP          [32] {mult, plus} of the jitter jump by 2 c k draws (c the partition stride), one-pixel tasks
//                    (ACC_REG) only: the block is SM_JUMP_BYTES longer there
#define RT_SMALL_MAX_SPHERES 8
#define RT_SMALL_MAX_SHAPES 16
#define RT_SMALL_MAX_MATERIALS 16
#define RT_SMALL_MAX_PIGMENTS 32
enum {
  SM_INVM = 0,
  SM_M = SM_INVM + RT_SMALL_MAX_SHAPES * 48,
  SM_ORIG = SM_M + RT_SMALL_MAX_SHAPES * 48,
  SM_PLANE2 = SM_ORIG + RT_SMALL_MAX_SHAPES * 4,
  SM_SHAPE_MAT = SM_PLANE2 + RT_SMALL_MAX_SHAPES / 2 * 32,
  SM_PIG = SM_SHAPE_MAT + RT_SMALL_MAX_SHAPES * 16,
  SM_PIG_STRIDE = 48,
  SM_BYTES = SM_PIG + RT_SMALL_MAX_PIGMENTS * SM_PIG_STRIDE,
  SM_JUMP = SM_BYTES,
  SM_JUMP_BYTES = 32 * 16
};
#ifndef RT_SMALL_THREADS
#define RT_SMALL_THREADS 256
#endif
#ifndef RT_SMALL_MINB
#define RT_SMALL_MINB 3
#endif

RT_DEV void stage_words(void* sh, const void* g, int bytes) {  // 4-byte granularity
  const uint32_t* src = reinterpret_cast<const uint32_t*>(g);
  uint32_t* dst = reinterpret_cast<uint32_t*>(sh);
  for (int i = threadIdx.x; i < bytes / 4; i += blockDim.x) dst[i] = __ldg(src + i);
}

// SM_INVM / SM_M layout from row-major [n][12] (see the table list above)
RT_DEV void stage_xf_pairs(void* sh, const float* g, int n_shapes) {
  float* dst = reinterpret_cast<float*>(sh);
  for (int i = threadIdx.x; i < n_shapes * 12; i += blockDim.x) {
    const int k = i % 12, src = k < 8 ? ((k & 1) << 2) + (k >> 1) : k;  // 0 4 1 5 2 6 3 7 8 9 10 11
    dst[i] = __ldg(g + (i - k) + src);
  }
}

// ---- shared memory by 32-bit window address ------------------------------------------------------
// On sm_100 the address an LDS takes is (cluster CTA id << 24) + offset, and the compiler re-derives
// that base (S2R SR_CgaCtaId + LEA, ~25 cycles of latency each time) at nearly every access when
// registers are short: ncu counted 11 such sequences per iteration of the drain loop on demo.txt, 6 %
// of the instruction stream.  The wavefront kernel therefore keeps ONE base address per warp that has
// been passed through a shuffle (not re-derivable) and addresses its work stack and the staged scene
// tables relative to it with explicit ld.shared / st.shared.
RT_DEV float4 lds4(uint32_t a) {  // read/write data (work stack): ordered against st.shared and __syncwarp
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
RT_DEV void sts4(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" :: "r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// tables that are constant once staged: no "memory" clobber, so loads may move across ordinary memory
// operations; volatile keeps them behind the __syncthreads() that ends the staging
RT_DEV float4 lds4c(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
RT_DEV int4 lds4ic(uint32_t a) {
  int4 v;
  asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
RT_DEV int ldsic(uint32_t a) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
RT_DEV ulonglong2 lds2u64c(uint32_t a) {
  ulonglong2 v;
  asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "r"(a));
  return v;
}

// Closest hit over a handful of shapes staged at `sb` (demo.txt: one sphere, two planes): World.ray_intersection
// (world.py:51-69) without a sweep / candidate list, every shape tested directly and without branches —
// with 32 different rays per warp some lane crosses every shape anyway.  Rays of the path tracer are
// unbounded (tmax = inf, ray.py:31), so only tmin is tested.  Spheres and planes keep separate minima
// (strict '<': the first of each kind wins a tie like world.py:62) and the rare sphere-vs-plane tie is
// resolved once at the end on the index in World.shapes.
// Both walks are unrolled to the SMALL capacity with one warp-uniform exit per shape (the counts are kernel
// parameters, read from the constant bank): no loop counter, and every table offset is an immediate off `sb`
// (spheres) or off the first plane's address (planes).  A runtime-bounded loop cost ~15 instructions of
// header per shape, as much as a plane test.
//
// The per-ray arithmetic runs partly on the paired FP32 pipe (fma.rn.f32x2, SASS FFMA2), on operands the staged
// tables hold as register pairs: rows 0 and 1 of a transform column by column (one packed FMA chain gives
// {x', y'} of a point or a direction), and the plane rows two planes at a time.  The ray's components enter as
// scalar broadcast operands.  Each half of a packed FMA is one fmaf and a packed product is one fp32 product,
// so every value is the same IEEE operation in the same association as in the scalar forms of rt_device.cuh
// (sphere_cross_rows, local_hit_rows, world_frame_rows): the image is the same bit for bit.
struct XfPairs {  // a SM_INVM / SM_M entry in registers
  f32x2 x, y, z, w;  // {r0.c, r1.c} for the columns c = x, y, z, w
  float4 r2;
};
RT_DEV XfPairs lds_xf(uint32_t a) {
  XfPairs m;
  const ulonglong2 p = lds2u64c(a), q = lds2u64c(a + 16);
  m.x = p.x; m.y = p.y; m.z = q.x; m.w = q.y;
  m.r2 = lds4c(a + 32);
  return m;
}
RT_DEV f32x2 bc2(float v) { return pk2(v, v); }  // a scalar broadcast operand of a packed instruction
// {x', y'} of M p + t (fmaf(r.x, p.x, fmaf(r.y, p.y, fmaf(r.z, p.z, r.w))) per row) and of M v
// (fmaf(r.x, v.x, fmaf(r.y, v.y, r.z * v.z)))
RT_DEV f32x2 xf_point01(const XfPairs& m, V3<float> p) { return fma2(m.x, bc2(p.x), fma2(m.y, bc2(p.y), fma2(m.z, bc2(p.z), m.w))); }
RT_DEV f32x2 xf_vec01(const XfPairs& m, V3<float> v) { return fma2(m.x, bc2(v.x), fma2(m.y, bc2(v.y), mul2(m.z, bc2(v.z)))); }
// sphere_cross_rows on a staged entry
RT_DEV bool sphere_cross_small(const XfPairs& M, const Ray<float>& r, float& tm, float& half) {
  const float4 r2 = M.r2;
  const f32x2 pxy = xf_point01(M, r.o), dxy = xf_vec01(M, r.d);
  float px, py, dx, dy;
  upk2(pxy, px, py); upk2(dxy, dx, dy);
  const float pz = fmaf(r2.x, r.o.x, fmaf(r2.y, r.o.y, fmaf(r2.z, r.o.z, r2.w)));
  const float dz = fmaf(r2.x, r.d.x, fmaf(r2.y, r.d.y, r2.z * r.d.z));
  const float a = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
  const float hb = fmaf(px, dx, fmaf(py, dy, pz * dz));
  const float inv = fast_rcp(a);
  const float s = hb * inv;
  float qx, qy;
  upk2(fma2(dxy, bc2(-s), pxy), qx, qy);
  const float qz = fmaf(-s, dz, pz);
  const float w = (1.0f - fmaf(qx, qx, fmaf(qy, qy, qz * qz))) * inv;
  tm = -s;
  half = fast_sqrt(fmaxf(w, 0.0f));
  return w > 0.0f;
}
// local_hit_rows and world_frame_rows on staged entries
RT_DEV LocalHit<float> local_hit_rows(const XfPairs& M, const Ray<float>& r, float t) {
  LocalHit<float> L;
  V3<float> o;
  upk2(xf_point01(M, r.o), o.x, o.y);
  upk2(xf_vec01(M, r.d), L.d.x, L.d.y);
  o.z = fmaf(r.o.x, M.r2.x, fmaf(r.o.y, M.r2.y, fmaf(r.o.z, M.r2.z, M.r2.w)));
  L.d.z = fmaf(r.d.x, M.r2.x, fmaf(r.d.y, M.r2.y, r.d.z * M.r2.z));
  L.hp = o + t * L.d;
  return L;
}
RT_DEV void world_frame_rows(const XfPairs& I, const XfPairs& M, const LocalHit<float>& L, bool sphere, V3<float>& point, V3<float>& normal) {
  upk2(xf_point01(M, L.hp), point.x, point.y);
  point.z = fmaf(L.hp.x, M.r2.x, fmaf(L.hp.y, M.r2.y, fmaf(L.hp.z, M.r2.z, M.r2.w)));
  V3<float> n;
  if (sphere) n = (dot(L.hp, L.d) < 0.f) ? L.hp : -L.hp;  // shapes.py:45-54
  else n = mk3<float>(0.f, 0.f, (L.d.z < 0.f) ? 1.f : -1.f);
  float i0x, i1x, i0y, i1y, i0z, i1z;
  upk2(I.x, i0x, i1x); upk2(I.y, i0y, i1y); upk2(I.z, i0z, i1z);
  n = mk3<float>(fmaf(n.x, i0x, fmaf(n.y, i1x, n.z * I.r2.x)),   // transpose of the inverse
                 fmaf(n.x, i0y, fmaf(n.y, i1y, n.z * I.r2.y)),
                 fmaf(n.x, i0z, fmaf(n.y, i1z, n.z * I.r2.z)));
  normal = normalize(n);
}
RT_DEV void closest_small(uint32_t sb, int n_spheres, int n_shapes, const Ray<float>& r, int origin, float& best_t, int& best) {
  const float inf = Num<float>::inf();
  float ts = inf, tp = inf;
  int is = -1, ip = -1;
#pragma unroll
  for (int i = 0; i < RT_SMALL_MAX_SPHERES; ++i) {
    if (i >= n_spheres) break;
    float tm, half;
    bool ok = sphere_cross_small(lds_xf(sb + SM_INVM + 48 * i), r, tm, half);
    const float t1 = tm - half;
    float t = (t1 > r.tmin) ? t1 : tm + half;   // the first root beyond tmin, shapes.py:112-119
    if (i == origin) { t = 2.0f * tm; ok = true; }  // see sphere_t_at
    if (ok && t > r.tmin && t < ts) { ts = t; is = i; }
  }
  // plane k is shape n_spheres + k; planes 2j and 2j + 1 go through one packed chain
  const int n_planes = n_shapes - n_spheres, porigin = origin - n_spheres;
#pragma unroll
  for (int j = 0; j < RT_SMALL_MAX_SHAPES / 2; ++j) {
    if (2 * j >= n_planes) break;
    const ulonglong2 p = lds2u64c(sb + SM_PLANE2 + 32 * j), q = lds2u64c(sb + SM_PLANE2 + 32 * j + 16);
    float oz[2], dz[2];
    upk2(fma2(p.x, bc2(r.o.x), fma2(p.y, bc2(r.o.y), fma2(q.x, bc2(r.o.z), q.y))), oz[0], oz[1]);
    upk2(fma2(p.x, bc2(r.d.x), fma2(p.y, bc2(r.d.y), mul2(q.x, bc2(r.d.z)))), dz[0], dz[1]);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int k = 2 * j + h;
      if (k >= n_planes) break;
      const float t = -oz[h] * fast_rcp(dz[h]);
      if (!(fabsf(dz[h]) < 1e-5f) && t > r.tmin && t < tp && k != porigin) { tp = t; ip = k; }
    }
  }
  if (ip >= 0) ip += n_spheres;
  bool plane = tp < ts;
  if (tp == ts && ip >= 0 && is >= 0) plane = ldsic(sb + SM_ORIG + 4 * ip) < ldsic(sb + SM_ORIG + 4 * is);
  best_t = plane ? tp : ts;
  best = plane ? ip : is;
}

// Pigment.get_color (materials.py:58, :70-82, :96-100) from a staged 48-byte record
RT_DEV V3<float> pigment_color_small(uint32_t pa, float u, float v) {
  const int4 h = lds4ic(pa);
  const float4 q = lds4c(pa + 16);
  if (h.x == RT_PIGMENT_UNIFORM) return mk3<float>(q.x, q.y, q.z);
  const float4 w = lds4c(pa + 32);
  if (h.x == RT_PIGMENT_CHECKERED) {
    const int iu = __float2int_rd(u * (float)h.y), iv = __float2int_rd(v * (float)h.y);
    return (((iu ^ iv) & 1) == 0) ? mk3<float>(q.x, q.y, q.z) : mk3<float>(q.w, w.x, w.y);
  }
  int col = (int)(u * (float)h.z), row = (int)(v * (float)h.w);
  col = min(max(col, 0), h.z - 1);
  row = min(max(row, 0), h.w - 1);
  const cudaTextureObject_t tex = ((unsigned long long)__float_as_uint(w.w) << 32) | (unsigned long long)__float_as_uint(w.z);
  const float4 t = fetch_texel(tex, col + 0.5f, row + 0.5f);
  return mk3<float>(t.x, t.y, t.z);
}

// Primary ray of the path tracer's warp kernels.  Same formulas as primary_ray<T> (imagetracer.py:48-58,
// :88-93, camera.py) in fp64, with the five divisions by width / height / S / 0xFFFFFFFF replaced by
// multiplications with the host-rounded reciprocals: a correctly rounded fp64 division costs ~30
// instructions and a sample needs six of them.  The fp64 values differ from the reference's by at most an
// ulp (1e-16), so the fp32 ray they round to is the reference's ray except when a coordinate sits within
// 1e-16 of an fp32 rounding boundary (~1e-8 of the rays) — immaterial for this renderer, whose parity is
// statistical; the deterministic renderers, the replay mode and the ray probes keep the divisions.
RT_DEV Ray<float> primary_ray_mul(const RenderArgs& a, double inv_w, double inv_h, double inv_s, int col, int row, int s, Pcg& aa) {
  double up = 0.5, vp = 0.5;
  if (a.S > 0) {
    const int ir = a.S <= 1024 ? (int)(((float)s + 0.5f) * (float)inv_s) : s / a.S;  // s / S, exact (s < S^2 <= 2^20)
    const int ic = s - ir * a.S;
    const double r1 = (double)pcg_random(aa) * (1.0 / 4294967295.0);
    const double r2 = (double)pcg_random(aa) * (1.0 / 4294967295.0);
    up = ((double)ic + r1) * inv_s;
    vp = ((double)ir + r2) * inv_s;
  }
  const double u = ((double)col + up) * inv_w;
  const double v = 1.0 - ((double)row + vp) * inv_h;
  V3<double> o, d;
  camera_fire_f64(a.cam, u, v, o, d);
  Ray<float> r;
  r.o = cast3<float>(o);
  r.d = cast3<float>(d);
  r.tmin = 1.0e-5f;
  r.tmax = Num<float>::inf();
  return r;
}

RT_DEV int own_stratum(const RenderArgs& a, int ls) {
  return (a.part_mode == RT_PART_SPP && a.part_count > 1) ? a.part_rank + ls * a.part_count : ls;
}

// SMALL: scenes of at most 8 spheres (demo.txt): the sweep is not unrolled and the kernel is held to
// 80 registers so that three CTAs (24 warps) fit an SM; large scenes are FMA-bound in the unrolled
// sweep and keep the 128-register budget.
// ACC: how per-pixel sums are kept while a task is in flight.
//   ACC_REG   one pixel per task: lane-private registers, one warp reduction at the end
//   ACC_LANES 2..8 pixels per task: acc[slot][channel][lane] in shared memory — every lane adds into
//             its own column (no conflicts, no atomics), reduced over lanes at the end
//   ACC_SEG   more pixels per task: segmented warp scan over the lanes of a record, then one
//             shared-memory atomic per record
enum { ACC_REG = 0, ACC_LANES = 1, ACC_SEG = 2 };
#define RT_ACC_LANES_MAX_GROUP 8

// ERR: error-map instantiation (see err_batch_add): tasks over ea.pix_list when set, and instead of the image
// every pixel's pass mean and SE^2 go to ea.err_mean / ea.err_var; the slot of a scatter record is then the batch.
template <bool SHAPES_SMEM, int ACC, bool SMALL, bool ERR = false>
__global__ void __launch_bounds__(SMALL ? RT_SMALL_THREADS : RT_WARP_MAX_THREADS, SMALL ? RT_SMALL_MINB : 2)
k_pt_warp(const __grid_constant__ SceneView<float> sc, const __grid_constant__ RenderArgs a,
          const __grid_constant__ WarpCfg cfg, const __grid_constant__ ErrArgs ea) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned FULL = 0xffffffffu;
  const int warp = threadIdx.x >> 5;
  ScanSrc<float> src = global_src<float>(sc);
  if (SMALL) {
    stage_xf_pairs(smem_raw + SM_INVM, sc.invm, sc.n_shapes);
    stage_xf_pairs(smem_raw + SM_M, sc.m, sc.n_shapes);
    for (int i = threadIdx.x; i < RT_SMALL_MAX_SHAPES * 4; i += blockDim.x) {  // {x, x', y, y', z, z', w, w'} per plane pair
      const int k = sc.n_spheres + 2 * (i >> 3) + (i & 1);
      reinterpret_cast<float*>(smem_raw + SM_PLANE2)[i] = k < sc.n_shapes ? __ldg(sc.invm + 12 * k + 8 + ((i & 7) >> 1)) : 0.f;
    }
    stage_words(smem_raw + SM_ORIG, sc.orig, sc.n_shapes * 4);
    for (int i = threadIdx.x; i < sc.n_shapes; i += blockDim.x) {
      const DevMaterial& mt = sc.materials[sc.material[i]];
      reinterpret_cast<int4*>(smem_raw + SM_SHAPE_MAT)[i] = make_int4(mt.brdf_kind, mt.brdf_pigment, mt.emitted_pigment, mt.flags);
    }
    for (int i = threadIdx.x; i < sc.n_pigments; i += blockDim.x) {
      const DevPigment& pg = sc.pigments[i];
      float4* o = reinterpret_cast<float4*>(smem_raw + SM_PIG + i * SM_PIG_STRIDE);
      o[0] = make_float4(__int_as_float(pg.kind), __int_as_float(pg.steps), __int_as_float(pg.tex_w), __int_as_float(pg.tex_h));
      o[1] = make_float4(pg.c1[0], pg.c1[1], pg.c1[2], pg.c2[0]);
      o[2] = make_float4(pg.c2[1], pg.c2[2], __uint_as_float((uint32_t)pg.tex), __uint_as_float((uint32_t)((unsigned long long)pg.tex >> 32)));
    }
    if (ACC == ACC_REG && threadIdx.x < 32) {  // x -> mult x + plus = LCG^(2 c k), composed from a.jump
      const unsigned long long c = (a.part_mode == RT_PART_SPP && a.part_count > 1) ? (unsigned long long)a.part_count : 1ull;
      uint64_t d = 2ull * c * threadIdx.x, mult = 1, plus = 0;
      while (d != 0) {
        const int b = __ffsll((long long)d) - 1;
        mult = a.jump.mult[b] * mult;
        plus = a.jump.mult[b] * plus + a.jump.plus[b];
        d &= d - 1;
      }
      reinterpret_cast<ulonglong2*>(smem_raw + SM_JUMP)[threadIdx.x] = make_ulonglong2(mult, plus);
    }
    __syncthreads();
  } else if (SHAPES_SMEM) {
    stage_bytes(smem_raw, sc.packed, (size_t)sc.n_pairs * 96 + (size_t)(sc.n_shapes - sc.n_spheres) * 48);
    __syncthreads();
    src.pairs = reinterpret_cast<const float4*>(smem_raw);
    src.planes = reinterpret_cast<const float*>(smem_raw) + 24 * (size_t)sc.n_pairs;
  }
  // lane index and the two shared-window addresses the loop lives on, each passed through a shuffle so
  // that they are values held (or spilled) instead of special-register sequences re-derived at every use
  const int lane0 = threadIdx.x & 31;
  const int lane = __shfl_sync(FULL, lane0, lane0);
  const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
  // (lane 0's value of a lane-dependent expression: a shuffle of a warp-uniform value would be folded away)
  const uint32_t sb = __shfl_sync(FULL, smem0 + (uint32_t)lane0, 0);  // staged scene tables (SMALL)
  const int wofs = (SMALL ? (int)SM_BYTES + (ACC == ACC_REG ? (int)SM_JUMP_BYTES : 0) : cfg.shape_bytes) + warp * cfg.per_warp_bytes;
  const uint32_t wb = __shfl_sync(FULL, smem0 + (uint32_t)(wofs + lane0), 0);  // this warp's record stack
  const uint32_t curb = wb + (uint32_t)cfg.cap * (uint32_t)sizeof(ScatterRec);  // the partly consumed record
  constexpr bool MULTI_SLOT = ACC != ACC_REG;
  int* slot_rays = reinterpret_cast<int*>(smem_raw + wofs + (size_t)(cfg.cap + 1) * sizeof(ScatterRec));  // [32], multi-pixel tasks + RT_HIT_RAY_COUNT
  float* acc = reinterpret_cast<float*>(slot_rays + 32);   // ACC_SEG: [32][3]; ACC_LANES: [G][3][32]
  // ERR: batch sums [32][3] behind the accumulator (ACC_REG has neither slot_rays nor acc: they go there)
  float* bsum = ACC == ACC_REG ? reinterpret_cast<float*>(slot_rays) : acc + (ACC == ACC_SEG ? 96 : 96 * cfg.group);
  const bool count_rays = a.out_hit != nullptr && a.hit_mode == RT_HIT_RAY_COUNT;

  const PixelMap pm = ERR ? make_pixel_map_list(a, ea) : make_pixel_map(a);
  const int N = a.num_of_rays;
  const int S2 = a.S > 0 ? a.S * a.S : 1;
  const int G = cfg.group, L = cfg.per_pixel;
  // x / N for 0 <= x <= 32 as a multiply-shift (exact for N <= 1024; beyond that x / N is 0 or 1)
  auto div_n = [&](int x) -> int { return cfg.n_magic ? (int)(((unsigned)x * cfg.n_magic) >> 16) : (x >= N ? 1 : 0); };
  const float inv_n = cfg.inv_n, inv_spp = cfg.inv_spp;
  // rays are counted per task from warp-uniform quantities (every lane holds the same sum)
  unsigned int n_rays = 0;
  bool overflow = false;

  while (true) {
    long long task = 0;
    if (lane == 0) task = (long long)atomicAdd(a.counters + CNT_TASK, 1ull);
    task = __shfl_sync(FULL, task, 0);
    if (task >= cfg.n_tasks) break;
    const long long p0 = task * G;
    // one pixel per task: the jitter stream is taken to the pixel's first draw once, lanes jump on by 2 s
    uint64_t aa_task = a.aa_state;
    if (ACC == ACC_REG && a.S > 0 && p0 < pm.n_pixels) {
      int col, row;
      if (ERR) locate_listed(pm, ea, p0, col, row);
      else pm.locate(p0, col, row);
      aa_task = pcg_jump(a.aa_state, 2ull * (unsigned long long)((long long)row * a.width + col) * S2, a.jump);
    }
    float sr = 0.f, sg = 0.f, sb_ = 0.f;  // lane-private sums (single-slot tasks)
    unsigned int task_rays = 0;           // warp-uniform
    const int task_prims = (int)min((long long)G, pm.n_pixels - p0) * L;  // primaries of this task
    if (MULTI_SLOT) {
      if (ACC == ACC_SEG) { for (int i = lane; i < 96; i += 32) acc[i] = 0.f; }
      else { for (int i = 0; i < 3 * cfg.group; ++i) acc[i * 32 + lane] = 0.f; }
      slot_rays[lane] = 0;
      __syncwarp();
    }
    if (ERR) {
      for (int i = lane; i < 96; i += 32) bsum[i] = 0.f;
      __syncwarp();
    }

    // All samples of the task start first (cfg.rounds warp-wide primary iterations pushing onto one
    // stack), then the stack drains once: the partially filled iterations at the end of a drain are
    // paid once per task instead of once per 32 samples.
    {
      int top = 0, cur_rem = 0, cur_done = 0;
      int round = 0;
      bool primary_phase = true;
      while (true) {
        // ---------------- pick this lane's ray
        bool active;
        int slot = 0, depth = 0, seg_start = lane, origin = -1;
        V3<float> thr = mk3<float>(1.f, 1.f, 1.f);
        Ray<float> ray;
        Pcg rng;
        long long pix = 0;
        bool last_of_pixel = false;
        int rslot = 0;  // ERR: the slot field of this ray's records, the batch (`slot` stays the pixel in the task)
        if (primary_phase) {
          // SMALL one-pixel tasks: sample ls = 32 round + lane has stratum own_stratum(32 round) + c lane (c the
          // partition stride), so its jitter state J_2s(aa_task) is the lane's table entry applied to one
          // warp-uniform jump per round (affine maps mod 2^64 compose exactly)
          uint64_t aa_round = 0;
          if (SMALL && ACC == ACC_REG && a.S > 0) aa_round = pcg_jump(aa_task, 2ull * (unsigned)own_stratum(a, round * 32), a.jump);
          const int j = round * 32 + lane;
          slot = j / L;
          const int ls = j - slot * L;
          const long long p = p0 + slot;
          if (ERR) rslot = slot * ea.err_bpp + err_batch_of(ea, ls);
          active = (j < G * L) && (p < pm.n_pixels);
          task_rays += (unsigned)min(max(task_prims - round * 32, 0), 32);
          if (active) {
            int col, row;
            if (ERR) locate_listed(pm, ea, p, col, row);
            else pm.locate(p, col, row);
            pix = (long long)row * a.width + col;
            const int s = own_stratum(a, ls);
            const unsigned long long k = (unsigned long long)pix * S2 + s;
            Pcg aa;
            aa.inc = a.aa_inc;
            if (SMALL && ACC == ACC_REG) {
              const ulonglong2 jl = lds2u64c(sb + SM_JUMP + 16 * lane);
              aa.state = (a.S > 0) ? jl.x * aa_round + jl.y : 0;
            } else if (ACC == ACC_REG) aa.state = (a.S > 0) ? pcg_jump(aa_task, 2ull * (unsigned)s, a.jump) : 0;
            else aa.state = (a.S > 0) ? pcg_jump(a.aa_state, 2ull * k, a.jump) : 0;
            ray = primary_ray_mul(a, cfg.inv_w, cfg.inv_h, cfg.inv_s, col, row, s, aa);
            rng = pcg_seed(a.pt_state, (a.pt_inc >> 1) + k);
            last_of_pixel = (ls == L - 1);
          }
          if (ACC == ACC_SEG) seg_start = max(0, slot * L - round * 32);
        } else {
          const long long avail = (long long)cur_rem + (long long)top * N;
          if (avail == 0) break;
          const int take = (int)min(avail, 32ll);
          active = lane < take;
          task_rays += (unsigned)take;
          // the first `from_cur` lanes finish the partly consumed record, the others take whole records
          // off the top, N lanes each: one address per lane, one set of three broadcast LDS.128
          const int from_cur = min(cur_rem, take);
          const int jj = max(lane - from_cur, 0);
          const int r = div_n(jj);
          const bool on_cur = lane < from_cur;
          const int child = on_cur ? cur_done + lane : jj - r * N;
          if (ACC == ACC_SEG) seg_start = on_cur ? 0 : from_cur + r * N;
          const uint32_t ra = (on_cur || !active) ? curb : wb + (uint32_t)(top - 1 - r) * (uint32_t)sizeof(ScatterRec);
          ScatterRec rec;
          rec.a = lds4(ra); rec.b = lds4(ra + 16); rec.c = lds4(ra + 32);
          // bookkeeping, identical in all lanes
          const int rest = take - from_cur;
          const int full = div_n(rest), part = rest - full * N;
          cur_rem -= from_cur;
          cur_done += from_cur;
          __syncwarp();  // every lane has read its record
          int new_top = top - full;
          if (part > 0) {  // the next record is only partly consumed: it becomes `cur`
            new_top -= 1;
            if (lane < 3) sts4(curb + 16 * lane, lds4(wb + (uint32_t)new_top * (uint32_t)sizeof(ScatterRec) + 16 * lane));
            cur_rem = N - part;
            cur_done = part;
          }
          __syncwarp();
          top = new_top;
          if (active) {
            const int meta = __float_as_int(rec.a.w);
            slot = meta & 31;
            if (ERR) { rslot = slot; slot = (int)(((unsigned)rslot * ea.err_magic) >> 16); }  // the batch's pixel in the task
            depth = (meta >> 6) & 1023;
            origin = (int)((unsigned)meta >> 16);
            if (origin == 0xFFFF) origin = -1;
            thr = mk3<float>(rec.b.w, rec.c.x, rec.c.y);
            const uint64_t base = ((uint64_t)__float_as_uint(rec.c.w) << 32) | (uint64_t)__float_as_uint(rec.c.z);
            rng.state = child_stream(base, child);
            rng.inc = a.pt_inc;
            ray.o = mk3<float>(rec.a.x, rec.a.y, rec.a.z);
            ray.tmax = Num<float>::inf();
            const V3<float> nd = mk3<float>(rec.b.x, rec.b.y, rec.b.z);
            if (((meta >> 5) & 1) == RT_BRDF_DIFFUSE) {
              const float u1 = unit_from_u32((uint32_t)(rng.state >> 32));  // the two halves of the child's stream value
              const float u2 = unit_from_u32((uint32_t)rng.state);
              ray.d = diffuse_dir<float>(nd, u1, u2);
              ray.tmin = 1.0e-3f;
            } else {
              ray.d = nd;
              ray.tmin = 1e-5f;
            }
          }
        }

        // ---------------- trace + shade
        V3<float> contrib = mk3<float>(0.f, 0.f, 0.f);
        bool push = false;
        ScatterRec out;
        float best_t = Num<float>::inf();
        int best = -1;
        if (!SMALL && RT_WARP_SPLIT) {  // large scenes: the whole warp sweeps together, half-warps on different pairs
          if (!active) { ray.o = mk3<float>(0.f, 0.f, 0.f); ray.d = mk3<float>(0.f, 0.f, 0.f); ray.tmin = 0.f; ray.tmax = 0.f; }
          closest_all_warp(sc, src, ray, active, best_t, best, origin);
        }
        if (active) {
          if (SMALL) closest_small(sb, sc.n_spheres, sc.n_shapes, ray, origin, best_t, best);
          else if (!RT_WARP_SPLIT) closest_all_f32<true>(sc, src, ray, best_t, best, origin);
          const bool found = best >= 0;
          if (count_rays) {
            if (MULTI_SLOT) atomicAdd(&slot_rays[slot], 1);
          } else if (primary_phase) {  // (warp-uniform)
            if (last_of_pixel && a.out_hit)
              a.out_hit[pm.compact ? p0 + slot : pix] = !found ? -1 : (SMALL ? ldsic(sb + SM_ORIG + 4 * best) : sc.orig[best]);
          }
          if (!found) {
            contrib = mk3<float>(thr.x * cfg.bg[0], thr.y * cfg.bg[1], thr.z * cfg.bg[2]);
          } else {
            // The hit record is built lazily (rt_device.cuh local_hit / local_uv / world_frame): most rays
            // of a tree are its leaves, whose children render.py:100-101 cuts — for those only the emitted
            // colour matters, which for a uniform pigment needs no record at all.
            int brdf_kind, brdf_pig, emit_pig, mf;
            typename std::conditional<SMALL, XfPairs, Rows3>::type im;
            const bool sphere = best < sc.n_spheres;
            if (SMALL) {
              const int4 mt = lds4ic(sb + SM_SHAPE_MAT + 16 * best);
              brdf_kind = mt.x; brdf_pig = mt.y; emit_pig = mt.z; mf = mt.w;
            } else {
              const DevMaterial& mat = sc.materials[sc.material[best]];
              brdf_kind = mat.brdf_kind; brdf_pig = mat.brdf_pigment; emit_pig = mat.emitted_pigment; mf = mat.flags;
            }
            auto rows_of = [&](bool inverse) -> decltype(im) {
              if constexpr (SMALL) return lds_xf(sb + (inverse ? SM_INVM : SM_M) + 48 * best);
              else return rows_at((inverse ? sc.invm : sc.m) + 12 * (size_t)best);
            };
            auto pig_uniform = [&](int idx) -> V3<float> {
              if (SMALL) { const float4 q = lds4c(sb + SM_PIG + idx * SM_PIG_STRIDE + 16); return mk3<float>(q.x, q.y, q.z); }
              return pig_c1<float>(sc.pigments[idx]);
            };
            auto pig_at = [&](int idx, float u, float v) -> V3<float> {
              if (SMALL) return pigment_color_small(sb + SM_PIG + idx * SM_PIG_STRIDE, u, v);
              return pigment_color<float>(sc.pigments, idx, u, v);
            };
            float u = 0.f, v = 0.f;
            if (depth >= a.max_depth) {
              // every child would come back BLACK, so neither the roulette draw (render.py:116-123) nor
              // the BRDF colour can change the result: emitted radiance only
              if (!(mf & MAT_EMIT_BLACK)) {
                if (mf & MAT_UV_EMIT) local_uv<float>(local_hit_rows(rows_of(true), ray, best_t), sphere, u, v);
                contrib = mul3(thr, (mf & MAT_UV_EMIT) ? pig_at(emit_pig, u, v) : pig_uniform(emit_pig));
              }
            } else {
              const bool scatters = !(mf & MAT_NO_SCATTER);
              LocalHit<float> lh;
              if (scatters || (mf & MAT_USES_UV)) { im = rows_of(true); lh = local_hit_rows(im, ray, best_t); }
              if (mf & MAT_USES_UV) local_uv<float>(lh, sphere, u, v);
              if (!(mf & MAT_EMIT_BLACK))
                contrib = mul3(thr, (mf & MAT_UV_EMIT) ? pig_at(emit_pig, u, v) : pig_uniform(emit_pig));
              if (scatters) {
                V3<float> hit_color = (mf & MAT_UV_BRDF) ? pig_at(brdf_pig, u, v) : pig_uniform(brdf_pig);
                const float lum = max3(hit_color);
                bool go_on = true;
                if (depth >= a.rr_limit) {  // render.py:116-123
                  const float q = fmaxf(0.05f, 1.f - lum);
                  if (pcg_random_float<float>(rng) > q) hit_color = fast_rcp(1.f - q) * hit_color;
                  else go_on = false;
                }
                if (go_on && lum > 0.f) {
                  push = true;
                  V3<float> point, normal;
                  // (SMALL reloads the inverse: held across the shading above, its 12 registers made ptxas spill
                  // loop state at the 80-register cap)
                  world_frame_rows(SMALL ? rows_of(true) : im, rows_of(false), lh, sphere, point, normal);
                  const V3<float> nd = (brdf_kind == RT_BRDF_DIFFUSE) ? normal : specular_dir<float>(ray.d, normal);
                  const V3<float> w = inv_n * mul3(thr, hit_color);
                  out.a = make_float4(point.x, point.y, point.z,
                                      __int_as_float((ERR ? rslot : slot) | (brdf_kind << 5) | ((depth + 1) << 6) |
                                                     ((best < 0xFFFF ? best : 0xFFFF) << 16)));
                  out.b = make_float4(nd.x, nd.y, nd.z, w.x);
                  out.c = make_float4(w.y, w.z, __uint_as_float((uint32_t)rng.state), __uint_as_float((uint32_t)(rng.state >> 32)));
                }
              }
            }
          }
        }

        // ---------------- accumulate
        if (ERR) err_batch_add(bsum, rslot, active, contrib, lane);
        if (ACC == ACC_SEG) {
          // lanes of one record (or one pixel, for primaries) are contiguous: segmented scan
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const float r = __shfl_up_sync(FULL, contrib.x, d);
            const float g = __shfl_up_sync(FULL, contrib.y, d);
            const float b = __shfl_up_sync(FULL, contrib.z, d);
            if (lane - d >= seg_start) { contrib.x += r; contrib.y += g; contrib.z += b; }
          }
          const int next_start = __shfl_down_sync(FULL, seg_start, 1);
          const bool tail = (lane == 31) || (next_start != seg_start);
          if (active && tail && (contrib.x != 0.f || contrib.y != 0.f || contrib.z != 0.f)) {
            atomicAdd(&acc[3 * slot + 0], contrib.x);
            atomicAdd(&acc[3 * slot + 1], contrib.y);
            atomicAdd(&acc[3 * slot + 2], contrib.z);
          }
        } else if (ACC == ACC_LANES) {
          if (active) {  // this lane's own column of the pixel's accumulator: no other lane touches it
            float* col = acc + (3 * slot) * 32 + lane;
            col[0] += contrib.x; col[32] += contrib.y; col[64] += contrib.z;
          }
        } else {
          sr += contrib.x; sg += contrib.y; sb_ += contrib.z;
        }

        // ---------------- push the new records: one ballot gives every lane its slot
        const unsigned pmask = __ballot_sync(FULL, push);
        const int npush = __popc(pmask);
        if (top + npush > cfg.cap) {
          overflow = true;
        } else {
          if (push) {
            const uint32_t pa = wb + (uint32_t)(top + __popc(pmask & ((1u << lane) - 1u))) * (uint32_t)sizeof(ScatterRec);
            sts4(pa, out.a); sts4(pa + 16, out.b); sts4(pa + 32, out.c);
          }
          top += npush;
        }
        __syncwarp();
        if (primary_phase && ++round >= cfg.rounds) primary_phase = false;
      }
    }
    n_rays += task_rays;

    // ---------------- write the pixels of this task
    if (ERR && ACC == ACC_SEG) {
      __syncwarp();
      for (int g = 0; g < G && p0 + g < pm.n_pixels; ++g)
        err_store(ea, L, bsum, g, p0 + g, mk3<float>(acc[3 * g] * inv_spp, acc[3 * g + 1] * inv_spp, acc[3 * g + 2] * inv_spp), lane);
      __syncwarp();
    } else if (ACC == ACC_SEG) {
      __syncwarp();
      const long long p = p0 + lane;
      if (lane < G && p < pm.n_pixels) {
        int col, row;
        pm.locate(p, col, row);
        store_pixel<float>(a, pm.at(p, col, row),
                           mk3<float>(acc[3 * lane] * inv_spp, acc[3 * lane + 1] * inv_spp, acc[3 * lane + 2] * inv_spp));
        if (count_rays) a.out_hit[pm.at(p, col, row)] = slot_rays[lane];
      }
      __syncwarp();
    } else if (ACC == ACC_LANES) {
      __syncwarp();
      for (int g = 0; g < G; ++g) {
        float r = acc[(3 * g) * 32 + lane], gr = acc[(3 * g + 1) * 32 + lane], b = acc[(3 * g + 2) * 32 + lane];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
          r += __shfl_xor_sync(FULL, r, d);
          gr += __shfl_xor_sync(FULL, gr, d);
          b += __shfl_xor_sync(FULL, b, d);
        }
        const long long p = p0 + g;
        if (ERR) {
          if (p < pm.n_pixels) err_store(ea, L, bsum, g, p, mk3<float>(r * inv_spp, gr * inv_spp, b * inv_spp), lane);
        } else if (lane == 0 && p < pm.n_pixels) {
          int col, row;
          pm.locate(p, col, row);
          store_pixel<float>(a, pm.at(p, col, row), mk3<float>(r * inv_spp, gr * inv_spp, b * inv_spp));
          if (count_rays) a.out_hit[pm.at(p, col, row)] = slot_rays[g];
        }
      }
      __syncwarp();
    } else {
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        sr += __shfl_xor_sync(FULL, sr, d);
        sg += __shfl_xor_sync(FULL, sg, d);
        sb_ += __shfl_xor_sync(FULL, sb_, d);
      }
      if (ERR) {
        if (p0 < pm.n_pixels) {
          __syncwarp();  // the batch sums of the task are complete
          err_store(ea, L, bsum, 0, p0, mk3<float>(sr * inv_spp, sg * inv_spp, sb_ * inv_spp), lane);
        }
        __syncwarp();
      } else if (lane == 0 && p0 < pm.n_pixels) {
        int col, row;
        pm.locate(p0, col, row);
        store_pixel<float>(a, pm.at(p0, col, row), mk3<float>(sr * inv_spp, sg * inv_spp, sb_ * inv_spp));
        if (count_rays) a.out_hit[pm.at(p0, col, row)] = (int)task_rays;
      }
    }
  }
  if (overflow) atomicExch(a.counters + CNT_OVERFLOW, 1ull);
  if (lane == 0 && n_rays) atomicAdd(a.counters + CNT_CLOSEST, (unsigned long long)n_rays);
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(a.counters + CNT_SAMPLES, cfg.n_samples);
}

template <bool ERR = false>
inline cudaError_t launch_pt_warp_impl(const SceneView<float>& sc, const RenderArgs& a, cudaStream_t st,
                                       int sm_count, LaunchInfo* info, const char** why_not, ErrArgs ea = ErrArgs()) {
  PixelMap pm = ERR ? make_pixel_map_list(a, ea) : make_pixel_map(a);
  const int S2 = a.S > 0 ? a.S * a.S : 1;
  int L = S2;
  if (a.part_mode == RT_PART_SPP && a.part_count > 1)
    L = a.part_rank < S2 ? (S2 - a.part_rank + a.part_count - 1) / a.part_count : 0;
  if (pm.n_pixels == 0 || L == 0) return cudaSuccess;
  if (a.num_of_rays < 1) { *why_not = "num_of_rays must be >= 1"; return cudaErrorInvalidValue; }
  if (a.max_depth >= 1023) { *why_not = "max_depth >= 1023 is not supported by the warp variant (use mega)"; return cudaErrorInvalidValue; }
  WarpCfg cfg;
  cfg.per_pixel = L;
  // Samples per task: all strata of one pixel when there are at least 32 of them (demo.txt at 64 spp:
  // 64-sample tasks, lane-private sums), otherwise as many pixels as make one warp-full of samples.
  size_t shape_bytes = (size_t)sc.n_pairs * 96 + (size_t)(sc.n_shapes - sc.n_spheres) * 48;
  const bool shapes_smem = shape_bytes > 0 && shape_bytes <= 64 * 1024;
  const bool small = sc.n_shapes > 0 && sc.n_spheres <= RT_SMALL_MAX_SPHERES && sc.n_shapes <= RT_SMALL_MAX_SHAPES &&
                     sc.n_materials <= RT_SMALL_MAX_MATERIALS && sc.n_pigments <= RT_SMALL_MAX_PIGMENTS;
  // (multi-pixel tasks, L < 32: 32 samples per task keep the accumulator columns small enough for three
  // resident blocks per SM — measured on demo.txt split over 8 GPUs: 50.9 vs 41.4 Grays/s per GPU)
  int want = 32;
#ifdef RT_TUNING  // tuning builds only (-DRT_TUNING): samples per multi-pixel task, clamped to what the kernel supports
  if (const char* env = getenv("RT_WARP_WANT")) want = std::min(std::max(atoi(env), 1), 256);
#endif
  if (L >= 32) cfg.group = 1;
  else if (L >= 4) cfg.group = (want + L - 1) / L < RT_ACC_LANES_MAX_GROUP ? (want + L - 1) / L : RT_ACC_LANES_MAX_GROUP;
  else cfg.group = 32 / L;
  if (cfg.group * L > 32 && !small) cfg.group = 32 / L > 0 ? 32 / L : 1;
  cfg.rounds = (cfg.group * L + 31) / 32;
  cfg.n_tasks = (pm.n_pixels + cfg.group - 1) / cfg.group;
  // stack capacity: every primary of the task may leave one level-1 record, and at most ~32 records
  // per deeper tree level are alive at any time (DESIGN.md §5.1); with N == 1 a record is replaced
  // by at most one record
  const long long prims = (long long)cfg.rounds * 32;
  long long cap = a.num_of_rays == 1 ? prims + 32 : prims + 32ll * (long long)a.max_depth;
  if (cap < 64) cap = 64;
  int acc_mode = cfg.group == 1 ? ACC_REG : (cfg.group <= RT_ACC_LANES_MAX_GROUP ? ACC_LANES : ACC_SEG);
  cfg.shape_bytes = small ? (int)SM_BYTES + (acc_mode == ACC_REG ? (int)SM_JUMP_BYTES : 0) : (shapes_smem ? (int)((shape_bytes + 15) / 16 * 16) : 0);
  const size_t limit = 200 * 1024;
  int warps = (small ? RT_SMALL_THREADS : RT_WARP_MAX_THREADS) / 32;
  size_t per_warp = 0, smem = 0;
  // (the accumulator choice below sums a pixel's samples in a different order per mode, so it is made on the
  // footprint without the batch sums: the ERR instantiation then stores the plain kernel's image bit for bit)
  bool with_err = false;
  auto footprint = [&](int mode, int w, size_t& pw) {
    pw = (size_t)(cap + 1) * sizeof(ScatterRec);
    if (mode == ACC_SEG) pw += 32 * sizeof(int) + 96 * sizeof(float);
    if (mode == ACC_LANES) pw += 32 * sizeof(int) + (size_t)cfg.group * 96 * sizeof(float);
    if (with_err) pw += 96 * sizeof(float);  // batch sums
    return cfg.shape_bytes + pw * w;
  };
  // The accumulator columns of ACC_LANES cost 384 B per pixel and warp; where that takes a resident
  // block away from the SM (demo.txt split over 4 or 8 GPUs: 2 blocks instead of 3, -25 % throughput)
  // the segmented-scan accumulators (ACC_SEG, 512 B per warp in all) are the better trade.
  if (acc_mode == ACC_LANES) {
    size_t pw_l, pw_s;
    const size_t sm_bytes = 227 * 1024;
    const size_t blocks_lanes = sm_bytes / (footprint(ACC_LANES, warps, pw_l) + 1024);
    const size_t blocks_seg = sm_bytes / (footprint(ACC_SEG, warps, pw_s) + 1024);
    const size_t by_threads = 2048 / (warps * 32), by_regs = small ? RT_SMALL_MINB : 2;
    if (std::min(std::min(blocks_seg, by_threads), by_regs) > std::min(std::min(blocks_lanes, by_threads), by_regs)) acc_mode = ACC_SEG;
#ifdef RT_TUNING
    if (const char* env = getenv("RT_WARP_ACC")) { const int m = atoi(env); if (m == ACC_LANES || m == ACC_SEG) acc_mode = m; }
#endif
  }
  with_err = ERR;
  for (;; warps >>= 1) {
    smem = footprint(acc_mode, warps, per_warp);
    if (smem <= limit || warps == 1) break;
  }
  if (smem > limit) { *why_not = "max_depth needs a deeper work stack than shared memory holds"; return cudaErrorInvalidValue; }
  cfg.cap = (int)cap;
  cfg.per_warp_bytes = (int)per_warp;
  for (int k = 0; k < 3; ++k) cfg.bg[k] = (float)a.background[k];
  cfg.inv_n = 1.0f / (float)a.num_of_rays;
  cfg.inv_spp = 1.0f / (float)S2;
  cfg.n_magic = a.num_of_rays <= 1024 ? (65536u + (unsigned)a.num_of_rays - 1u) / (unsigned)a.num_of_rays : 0u;
  cfg.n_samples = (unsigned long long)pm.n_pixels * (unsigned long long)L;
  cfg.inv_w = 1.0 / (double)a.width;
  cfg.inv_h = 1.0 / (double)a.height;
  cfg.inv_s = a.S > 0 ? 1.0 / (double)a.S : 1.0;
  ea.err_bpp = 32 / cfg.group;
  ea.err_magic = (65536u + (unsigned)ea.err_bpp - 1u) / (unsigned)ea.err_bpp;  // x / bpp for x < 32
  if (ERR && (a.S < 2 || cfg.group > RT_ACC_LANES_MAX_GROUP || L != S2)) {
    *why_not = "the error map needs samples_per_side >= 2 and no partition";
    return cudaErrorInvalidValue;
  }

  void (*kern)(const SceneView<float>, const RenderArgs, const WarpCfg, const ErrArgs);
#define RT_PICK(ACCM)                                                                   \
  (small ? k_pt_warp<true, ACCM, true, ERR> : (shapes_smem ? k_pt_warp<true, ACCM, false, ERR> : k_pt_warp<false, ACCM, false, ERR>))
  if (acc_mode == ACC_REG) kern = RT_PICK(ACC_REG);
  else if (acc_mode == ACC_LANES) kern = RT_PICK(ACC_LANES);
  else kern = RT_PICK(ACC_SEG);
#undef RT_PICK
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit);
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  long long blocks = (long long)per_sm * sm_count;  // persistent: every block stays resident
  long long needed = (cfg.n_tasks + warps - 1) / warps;
  if (blocks > needed) blocks = needed;
  kern<<<(unsigned)blocks, warps * 32, smem, st>>>(sc, a, cfg, ea);
  if (info) { info->n_launches += 1; info->variant = RT_VARIANT_WARP; }
  return cudaGetLastError();
}
