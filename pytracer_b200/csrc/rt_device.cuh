// rt_device.cuh — device restatement of the per-ray functions of the reference, templated on the
// arithmetic type T (float: production path-tracing arithmetic; double: bit-faithful path of the
// deterministic renderers, compiled without multiply-add fusion).
//
//   closest hit  World.ray_intersection   world.py:51-69     -> scan_*/finish_hit
//   any hit      World.is_point_visible   world.py:71-80     -> any_hit_*
//   shapes       Sphere / Plane           shapes.py:97-198
//   pigments     Pigment.get_color        materials.py:58,70-82,96-100
//   BRDFs        eval / scatter_ray       materials.py:129-196, ONB geometry.py:247-262
//   cameras      fire_ray                 camera.py:59-78,103-124; imagetracer.py:48-58
#pragma once
#include "rt_math.cuh"
#include "rt_pcg.cuh"
#include "../../include/rt_api.h"

// ---------------------------------------------------------------- device-side scene tables
struct DevPigment {
  int32_t kind, steps, tex_w, tex_h;
  cudaTextureObject_t tex;  // float4 texels, point filter (fp32 path)
  const double* texels64;   // same texels in fp64 (fp64 path)
  float c1[3], c2[3];
  double c1d[3], c2d[3];
};
struct DevMaterial {
  int32_t brdf_kind, brdf_pigment, emitted_pigment;
  int32_t flags;  // MAT_*: what shading this material can skip (set once by rt_scene_create)
  double threshold;
};
enum {
  MAT_UV_BRDF = 1,     // the BRDF pigment is not uniform: shading needs (u, v)
  MAT_UV_EMIT = 2,     // the emitted-radiance pigment is not uniform
  MAT_EMIT_BLACK = 4,  // emitted radiance is uniform black: the emitted term is zero
  MAT_NO_SCATTER = 8,  // the BRDF pigment is uniform with no positive channel: render.py:125 never scatters
  MAT_USES_UV = MAT_UV_BRDF | MAT_UV_EMIT
};
struct DevLight {
  double pos[3], color[3], radius;
};

// Shapes are stored sorted by kind: spheres [0, n_spheres) then planes [n_spheres, n_shapes), each
// group in World.shapes order; `orig` maps back to the index in World.shapes.  Within a group a
// strict '<' scan keeps the first shape on ties like world.py:62; across groups ties are resolved
// on `orig`, so the winner is the one the reference's single loop would pick.
template <typename T> struct SceneView {
  const T* invm;  // [n][12] inverse transforms, the only per-shape data the scan loops read
  const T* m;     // [n][12]
  const int32_t* orig;
  const int32_t* material;  // by sorted index
  const DevMaterial* materials;
  const DevPigment* pigments;
  const DevLight* lights;
  int32_t n_shapes, n_spheres, n_lights;
  // fp32 only: [n_pairs][24] element-interleaved sphere pairs followed by [n_planes][12] planes
  const float* packed;
  int32_t n_pairs;
  float gate_a;  // see pack_ray: sqrt(8 u) max_i |M_i|_F over the spheres

  int32_t n_materials, n_pigments;
  // sphere hierarchy (rt_bvh.cuh), used when accel != 0
  const float4* bvh_nodes;
  const int32_t* bvh_prims;
  int32_t accel;
  float gate_t;  // sqrt(8 u) max_i |t_i| (translation column of the inverse transforms)
};

template <typename T> struct Hit {
  int32_t idx;   // sorted index, -1 = miss
  T t;
  V3<T> point, normal;  // world space, normal normalised
  T u, v;
};

// ---------------------------------------------------------------- shape tests (t only)
// Sphere.ray_intersection shapes.py:97-121 up to the choice of the root; returns t, +inf = miss
// (a valid t is always < tmax <= inf, so the closest-hit scan needs a single compare).
template <typename T> RT_DEV T sphere_t(const T* im, const Ray<T>& r) {
  V3<T> o = xf_point(im, r.o);
  V3<T> d = xf_vec(im, r.d);
  T a = dot(d, d);
  T b = (T)2 * dot(o, d);
  T c = dot(o, o) - (T)1;
  T delta = b * b - (T)4 * a * c;
  if (delta <= (T)0) return Num<T>::inf();
  T sd = Num<T>::sqrt(delta);
  T den = (T)2 * a;
  T t1 = Num<T>::div(-b - sd, den);
  T t2 = Num<T>::div(-b + sd, den);
  if (t1 > r.tmin && t1 < r.tmax) return t1;
  if (t2 > r.tmin && t2 < r.tmax) return t2;
  return Num<T>::inf();
}

// Plane.ray_intersection shapes.py:163-174; only row 2 of the inverse transform is needed for t.
template <typename T> RT_DEV T plane_t(const T* im, const Ray<T>& r) {
  T oz = r.o.x * im[8] + r.o.y * im[9] + r.o.z * im[10] + im[11];
  T dz = r.d.x * im[8] + r.d.y * im[9] + r.d.z * im[10];
  if (Num<T>::abs(dz) < (T)1e-5) return Num<T>::inf();
  T t = Num<T>::div(-oz, dz);
  if (t <= r.tmin || t >= r.tmax) return Num<T>::inf();
  return t;
}

// world.py:62 keeps the FIRST shape of World.shapes on equal t; spheres are scanned before planes
// here, so a plane that ties with the current best sphere wins iff it came first in World.shapes.
// Out of line: ties are rare and the two global loads must not be hoisted into the scan loop.
static __device__ __noinline__ bool plane_wins_tie(const int32_t* __restrict__ orig, int plane, int best) {
  return orig[plane] < orig[best];
}

template <typename T>
RT_DEV void scan_planes(const T* __restrict__ xf, int begin, int end, int n_spheres,
                        const int32_t* __restrict__ orig, const Ray<T>& r, T& best_t, int& best) {
  for (int i = max(begin, n_spheres); i < end; ++i) {
    T t = plane_t(xf + 12 * (i - begin), r);
    if (t < best_t) { best_t = t; best = i; }
    else if (t == best_t && best >= 0 && best < n_spheres) {
      if (plane_wins_tie(orig, i, best)) { best_t = t; best = i; }
    }
  }
}

// Closest-hit scan over sorted shapes [begin, end) held at `xf` (xf[0] is shape `begin`); the data
// may live in shared or global memory.  All lanes walk the same shapes: loads are broadcasts.
// Start with best_t = +inf, best = -1.
template <typename T>
RT_DEV void scan_closest(const T* __restrict__ xf, int begin, int end, int n_spheres,
                         const int32_t* __restrict__ orig, const Ray<T>& r, T& best_t, int& best) {
  int s_end = min(end, n_spheres);
#pragma unroll 2
  for (int i = begin; i < s_end; ++i) {
    T t = sphere_t(xf + 12 * (i - begin), r);
    if (t < best_t) { best_t = t; best = i; }
  }
  scan_planes<T>(xf, begin, end, n_spheres, orig, r, best_t, best);
}

// shapes.py:133-151 / :191-198 — true as soon as one shape blocks the segment
template <typename T>
RT_DEV bool scan_any(const T* __restrict__ xf, int begin, int end, int n_spheres, const Ray<T>& r) {
  int s_end = min(end, n_spheres);
  for (int i = begin; i < s_end; ++i) {
    const T* im = xf + 12 * (i - begin);
    V3<T> o = xf_point(im, r.o);
    V3<T> d = xf_vec(im, r.d);
    T a = dot(d, d);
    T b = (T)2 * dot(o, d);
    T c = dot(o, o) - (T)1;
    T delta = b * b - (T)4 * a * c;
    if (delta <= (T)0) continue;
    T sd = Num<T>::sqrt(delta);
    T den = (T)2 * a;
    T t1 = Num<T>::div(-b - sd, den);
    T t2 = Num<T>::div(-b + sd, den);
    if ((r.tmin < t1 && t1 < r.tmax) || (r.tmin < t2 && t2 < r.tmax)) return true;
  }
  for (int i = max(begin, n_spheres); i < end; ++i) {
    const T* im = xf + 12 * (i - begin);
    T oz = r.o.x * im[8] + r.o.y * im[9] + r.o.z * im[10] + im[11];
    T dz = r.d.x * im[8] + r.d.y * im[9] + r.d.z * im[10];
    if (Num<T>::abs(dz) < (T)1e-5) continue;
    T t = Num<T>::div(-oz, dz);
    if (r.tmin < t && t < r.tmax) return true;
  }
  return false;
}

// ---------------------------------------------------------------- fp32 production scans
// Same mathematics as sphere_t<float> (shapes.py:97-121), arranged for the FMA pipe: the ray is
// taken to the sphere's frame with 18 FFMA, a, b/2 and c cost 9 more, delta/4 = (b/2)^2 - a c two:
// 29 FMA-pipe instructions and three broadcast LDS.128 per sphere, nothing else in the common case.
// Spheres are tested four at a time; the few whose line is crossed (delta > 0) go to a per-lane
// candidate list and only those get the sqrt / reciprocal / range tests after the sweep — so the
// sweep itself has one (rarely taken) branch per four spheres.
//
// Does the ray's line cross the sphere, and where: evaluated from the point of the line closest to the
// centre, q = o' - (o'.d' / a) d', instead of from the discriminant.  The line crosses iff |q|^2 < 1 and
// the roots are t = tm -+ half with tm = -(o'.d') / a, half = sqrt((1 - |q|^2) / a) — the same numbers as
// (-b -+ sqrt(delta)) / 2a (shapes.py:103-121), but delta/4 = (o'.d')^2 - a (|o'|^2 - 1) subtracts two
// terms of size a |o'|^2 to find something of size a: for a ray that starts 10^3 radii away its fp32 value
// is rounding noise (phantom hits on spheres the ray passes at a distance), while |q|^2 is formed from a
// vector of the size of the answer.  The sweep keeps the cheap discriminant as its gate; every decision
// about a sphere (closest hit, shadow test, hierarchy leaf) comes from here.
struct Rows3 {  // a 3x4 transform as three rows already in registers
  float4 r0, r1, r2;
};
RT_DEV Rows3 rows_at(const float* __restrict__ p) {
  Rows3 M;
  M.r0 = reinterpret_cast<const float4*>(p)[0];
  M.r1 = reinterpret_cast<const float4*>(p)[1];
  M.r2 = reinterpret_cast<const float4*>(p)[2];
  return M;
}
RT_DEV bool sphere_cross_rows(const Rows3& M, const Ray<float>& r, float& tm, float& half) {
  const float4 r0 = M.r0, r1 = M.r1, r2 = M.r2;
  const float px = fmaf(r0.x, r.o.x, fmaf(r0.y, r.o.y, fmaf(r0.z, r.o.z, r0.w)));
  const float py = fmaf(r1.x, r.o.x, fmaf(r1.y, r.o.y, fmaf(r1.z, r.o.z, r1.w)));
  const float pz = fmaf(r2.x, r.o.x, fmaf(r2.y, r.o.y, fmaf(r2.z, r.o.z, r2.w)));
  const float dx = fmaf(r0.x, r.d.x, fmaf(r0.y, r.d.y, r0.z * r.d.z));
  const float dy = fmaf(r1.x, r.d.x, fmaf(r1.y, r.d.y, r1.z * r.d.z));
  const float dz = fmaf(r2.x, r.d.x, fmaf(r2.y, r.d.y, r2.z * r.d.z));
  const float a = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
  const float hb = fmaf(px, dx, fmaf(py, dy, pz * dz));
  const float inv = fast_rcp(a);
  const float s = hb * inv;
  const float qx = fmaf(-s, dx, px), qy = fmaf(-s, dy, py), qz = fmaf(-s, dz, pz);
  const float w = (1.0f - fmaf(qx, qx, fmaf(qy, qy, qz * qz))) * inv;
  tm = -s;
  half = fast_sqrt(fmaxf(w, 0.0f));
  return w > 0.0f;  // false for a = 0 too (s is NaN): the reference's delta = b^2 = 0 is a miss as well
}
RT_DEV bool sphere_cross(const float* __restrict__ im, const Ray<float>& r, float& tm, float& half) {
  return sphere_cross_rows(rows_at(im), r, tm, half);
}

#define RT_CAND_CAP 16

// ---- packed sweep: two spheres per FFMA2 (Blackwell fma.rn.f32x2) -------------------------------
// The fp32 scan array stores spheres in PAIRS, element-interleaved: pair p holds, for each of the 12
// matrix entries, {entry of sphere 2p, entry of sphere 2p+1} — 24 floats = six LDS.128, each register
// pair of which is directly a packed operand.  The ray components enter as scalar broadcast operands
// (FFMA2 Rd, Ra.F32x2, Rb.F32, Rc.F32x2), so one sphere pair costs 30 packed FMA-pipe instructions
// instead of 58 scalar ones: issue slots per sphere drop from ~36 to ~19 and the register-bank
// pressure of three-source FFMAs disappears (a 64-bit operand always takes one word from each bank).
// An odd sphere count is padded with an all-zero record (a = 0, c = -1: delta = 0, never crossed).
typedef unsigned long long f32x2;
RT_DEV f32x2 pk2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
RT_DEV void upk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
RT_DEV f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
RT_DEV f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
RT_DEV f32x2 sub2(f32x2 a, f32x2 b) { f32x2 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
RT_DEV f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// The sweep's gate delta/4 = (o'.d')^2 - a (|o'|^2 - 1) > 0 is evaluated in fp32 and every decision about a
// sphere is then taken by sphere_cross on the spheres that pass, so the gate must not LOSE spheres: a
// symmetric rounding noise in delta would turn into a bias (spheres that pass by noise are thrown out again
// by sphere_cross, spheres that fail by noise are gone — every sphere would shrink by the noise band, and an
// image of small far spheres comes out measurably brighter).  The noise is dominated by the cancellation in
// o' = M o + t: |delta error| / a <~ 4 |o'| 5u (|M|_F |o| + |t|), at most 20u (|M|_F |o| + |t|)^2.  So the
// gate tests against a sphere of radius^2 1 + s with s = 8u (A |o| + T)^2, A = max |M_i|_F, T = max |t_i| over
// the scene (about four standard deviations of the observed noise; not a proof — the renderers whose hit
// index must be exact take the rigorous gate of rt_resolve_hybrid.cuh).  It costs nothing: the constant -1
// of the |o'|^2 - 1 chain becomes the per-ray value -(1 + s).
struct PackedRay {  // ray components as broadcast pairs (the compiler turns them into .F32 scalar operands)
  f32x2 ox, oy, oz, dx, dy, dz, k0;
};
RT_DEV PackedRay pack_ray(const Ray<float>& r, float gate_a, float gate_t) {
  PackedRay q;
  q.ox = pk2(r.o.x, r.o.x); q.oy = pk2(r.o.y, r.o.y); q.oz = pk2(r.o.z, r.o.z);
  q.dx = pk2(r.d.x, r.d.x); q.dy = pk2(r.d.y, r.d.y); q.dz = pk2(r.d.z, r.d.z);
  const float w = fmaf(gate_a, fast_sqrt(fmaf(r.o.x, r.o.x, fmaf(r.o.y, r.o.y, r.o.z * r.o.z))), gate_t);
  const float k = -fmaf(w, w, 1.0f);
  q.k0 = pk2(k, k);
  return q;
}

// delta/4 of both spheres of one pair (24 floats at `q`)
RT_DEV f32x2 pair_qdelta(const float4* __restrict__ q, const PackedRay& r) {
  const float4 v0 = q[0], v1 = q[1], v2 = q[2], v3 = q[3], v4 = q[4], v5 = q[5];
  const f32x2 m00 = pk2(v0.x, v0.y), m01 = pk2(v0.z, v0.w), m02 = pk2(v1.x, v1.y), m03 = pk2(v1.z, v1.w);
  const f32x2 m10 = pk2(v2.x, v2.y), m11 = pk2(v2.z, v2.w), m12 = pk2(v3.x, v3.y), m13 = pk2(v3.z, v3.w);
  const f32x2 m20 = pk2(v4.x, v4.y), m21 = pk2(v4.z, v4.w), m22 = pk2(v5.x, v5.y), m23 = pk2(v5.z, v5.w);
  const f32x2 px = fma2(m00, r.ox, fma2(m01, r.oy, fma2(m02, r.oz, m03)));
  const f32x2 py = fma2(m10, r.ox, fma2(m11, r.oy, fma2(m12, r.oz, m13)));
  const f32x2 pz = fma2(m20, r.ox, fma2(m21, r.oy, fma2(m22, r.oz, m23)));
  const f32x2 dx = fma2(m00, r.dx, fma2(m01, r.dy, mul2(m02, r.dz)));
  const f32x2 dy = fma2(m10, r.dx, fma2(m11, r.dy, mul2(m12, r.dz)));
  const f32x2 dz = fma2(m20, r.dx, fma2(m21, r.dy, mul2(m22, r.dz)));
  const f32x2 a = fma2(dx, dx, fma2(dy, dy, mul2(dz, dz)));
  const f32x2 hb = fma2(px, dx, fma2(py, dy, mul2(pz, dz)));
  const f32x2 c = fma2(px, px, fma2(py, py, fma2(pz, pz, r.k0)));
  return sub2(mul2(hb, hb), mul2(a, c));
}

// Sweeps sphere pairs [p0, p1) whose data starts at `pairs` (pairs[0] = pair `base`); crossed spheres
// are appended to cand[] (ring of RT_CAND_CAP; nc counts all of them) as sorted sphere indices.
template <bool UNROLL2 = true>
RT_DEV void sweep_pairs(const float4* __restrict__ pairs, int base, int p0, int p1, const PackedRay& r,
                        int* cand, int& nc) {
  int p = p0;
  if constexpr (!UNROLL2) {  // few spheres (e.g. demo.txt): one pair at a time keeps the register count low
#pragma unroll 1
    for (; p < p1; ++p) {
      float a0, a1;
      upk2(pair_qdelta(pairs + 6 * (p - base), r), a0, a1);
      if (fmaxf(a0, a1) > 0.0f) {
        if (a0 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p; ++nc; }
        if (a1 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p + 1; ++nc; }
      }
    }
  } else {
  for (; p + 2 <= p1; p += 2) {
    const float4* q = pairs + 6 * (p - base);
    float a0, a1, b0, b1;
    upk2(pair_qdelta(q, r), a0, a1);
    upk2(pair_qdelta(q + 6, r), b0, b1);
    if (fmaxf(fmaxf(a0, a1), fmaxf(b0, b1)) > 0.0f) {
      if (a0 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p; ++nc; }
      if (a1 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p + 1; ++nc; }
      if (b0 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p + 2; ++nc; }
      if (b1 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p + 3; ++nc; }
    }
  }
  if (p < p1) {
    float a0, a1;
    upk2(pair_qdelta(pairs + 6 * (p - base), r), a0, a1);
    if (a0 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p; ++nc; }
    if (a1 > 0.0f) { cand[nc & (RT_CAND_CAP - 1)] = 2 * p + 1; ++nc; }
  }
  }
}

// Two rays against the same pair data: the six LDS.128 of a pair feed 60 packed FMAs instead of 30,
// which halves the shared-memory wavefronts per FMA (broadcast LDS.128 = 2 wavefronts; at one ray per
// thread the shared-memory pipe runs at 80 % of the FMA pipe's pace and throttles it).
RT_DEV void pair_qdelta2(const float4* __restrict__ q, const PackedRay& r0, const PackedRay& r1, f32x2& qd0, f32x2& qd1) {
  const float4 v0 = q[0], v1 = q[1], v2 = q[2], v3 = q[3], v4 = q[4], v5 = q[5];
  const f32x2 m00 = pk2(v0.x, v0.y), m01 = pk2(v0.z, v0.w), m02 = pk2(v1.x, v1.y), m03 = pk2(v1.z, v1.w);
  const f32x2 m10 = pk2(v2.x, v2.y), m11 = pk2(v2.z, v2.w), m12 = pk2(v3.x, v3.y), m13 = pk2(v3.z, v3.w);
  const f32x2 m20 = pk2(v4.x, v4.y), m21 = pk2(v4.z, v4.w), m22 = pk2(v5.x, v5.y), m23 = pk2(v5.z, v5.w);
#define RT_QD(r, out)                                                                  \
  {                                                                                    \
    const f32x2 px = fma2(m00, r.ox, fma2(m01, r.oy, fma2(m02, r.oz, m03)));           \
    const f32x2 py = fma2(m10, r.ox, fma2(m11, r.oy, fma2(m12, r.oz, m13)));           \
    const f32x2 pz = fma2(m20, r.ox, fma2(m21, r.oy, fma2(m22, r.oz, m23)));           \
    const f32x2 dx = fma2(m00, r.dx, fma2(m01, r.dy, mul2(m02, r.dz)));                \
    const f32x2 dy = fma2(m10, r.dx, fma2(m11, r.dy, mul2(m12, r.dz)));                \
    const f32x2 dz = fma2(m20, r.dx, fma2(m21, r.dy, mul2(m22, r.dz)));                \
    const f32x2 a = fma2(dx, dx, fma2(dy, dy, mul2(dz, dz)));                          \
    const f32x2 hb = fma2(px, dx, fma2(py, dy, mul2(pz, dz)));                         \
    const f32x2 c = fma2(px, px, fma2(py, py, fma2(pz, pz, r.k0)));                    \
    out = sub2(mul2(hb, hb), mul2(a, c));                                              \
  }
  RT_QD(r0, qd0)
  RT_QD(r1, qd1)
#undef RT_QD
}

RT_DEV void sweep_pairs2(const float4* __restrict__ pairs, int base, int p0, int p1, const Ray<float>& ray0,
                         const Ray<float>& ray1, float gate_a, float gate_t, int* cand0, int& nc0, int* cand1, int& nc1) {
  // the broadcast pairs are rebuilt here from the scalar rays: the compiler turns them into scalar
  // (.F32) operands of FFMA2, so they cost no registers outside the loop
  const PackedRay r0 = pack_ray(ray0, gate_a, gate_t), r1 = pack_ray(ray1, gate_a, gate_t);
  for (int p = p0; p < p1; ++p) {
    f32x2 q0, q1;
    pair_qdelta2(pairs + 6 * (p - base), r0, r1, q0, q1);
    float a0, a1, b0, b1;
    upk2(q0, a0, a1);
    upk2(q1, b0, b1);
    if (fmaxf(fmaxf(a0, a1), fmaxf(b0, b1)) > 0.0f) {
      if (a0 > 0.0f) { cand0[nc0 & (RT_CAND_CAP - 1)] = 2 * p; ++nc0; }
      if (a1 > 0.0f) { cand0[nc0 & (RT_CAND_CAP - 1)] = 2 * p + 1; ++nc0; }
      if (b0 > 0.0f) { cand1[nc1 & (RT_CAND_CAP - 1)] = 2 * p; ++nc1; }
      if (b1 > 0.0f) { cand1[nc1 & (RT_CAND_CAP - 1)] = 2 * p + 1; ++nc1; }
    }
  }
}

// Warp-cooperative sweep for one ray per lane (the path tracer's layout).  A broadcast LDS.128 costs
// two shared-memory wavefronts, one per half-warp, whatever the two halves read — so the halves read
// DIFFERENT pairs: lanes 0-15 sweep the first half of the pair list, lanes 16-31 the second half, each
// lane for its own ray and for the ray of its partner lane (lane ^ 16, fetched with six shuffles).  Same
// FMA work per lane (two rays x half the pairs), half the shared-memory wavefronts per FMA.  After the
// sweep the partner's candidates are handed back with shuffles and merged in ascending sphere order.
// Must be called by all 32 lanes (idle lanes pass a zero ray: a = 0, delta = 0, never crossed);
// n_pairs is even (rt_scene_create pads the pair list).
RT_DEV void sweep_pairs_split(const float4* __restrict__ pairs, int n_pairs, const Ray<float>& mine, float gate_a, float gate_t,
                              int* cand, int& nc) {
  const unsigned FULL = 0xffffffffu;
  const bool hi = (threadIdx.x & 16) != 0;
  Ray<float> other;
  other.o.x = __shfl_xor_sync(FULL, mine.o.x, 16); other.o.y = __shfl_xor_sync(FULL, mine.o.y, 16);
  other.o.z = __shfl_xor_sync(FULL, mine.o.z, 16); other.d.x = __shfl_xor_sync(FULL, mine.d.x, 16);
  other.d.y = __shfl_xor_sync(FULL, mine.d.y, 16); other.d.z = __shfl_xor_sync(FULL, mine.d.z, 16);
  const int half = n_pairs >> 1;
  const int first = hi ? half : 0;
  int theirs[RT_CAND_CAP];
  int n_mine = 0, n_theirs = 0;
  sweep_pairs2(pairs, 0, first, first + half, mine, other, gate_a, gate_t, cand, n_mine, theirs, n_theirs);
  // hand the partner's candidates back; the low half's spheres come first in the merged list
  const int n_recv = __shfl_xor_sync(FULL, n_theirs, 16);
  int merged[RT_CAND_CAP];
  const int total = n_mine + n_recv;
  const int at_recv = hi ? 0 : n_mine, at_mine = hi ? n_recv : 0;
#pragma unroll
  for (int j = 0; j < RT_CAND_CAP; ++j) {
    const int v = __shfl_xor_sync(FULL, theirs[j], 16);
    if (j < n_recv && at_recv + j < RT_CAND_CAP) merged[at_recv + j] = v;
  }
  if (n_mine <= RT_CAND_CAP && n_recv <= RT_CAND_CAP && total <= RT_CAND_CAP) {
    for (int j = 0; j < n_mine; ++j) merged[at_mine + j] = cand[j];
    for (int j = 0; j < total; ++j) cand[j] = merged[j];
    nc = total;
  } else {
    nc = RT_CAND_CAP + 1;  // too many crossed spheres for the lists: resolve_candidates does a plain pass
  }
}

// Exact roots for the crossed spheres only, from the plain [n][12] array in global memory (a few per
// ray: L1/L2 hits).  Ascending index + strict '<' keeps the first shape on ties (world.py:62).
//
// `origin` = sorted index of the shape the ray starts on (-1: none).  A ray that starts ON a sphere
// has c = |o|^2 - 1 = 0: its roots are t = 0 (never inside (tmin, tmax): the fp64 reference gets
// ~1e-16 there) and t = -b/a.  In fp32 c is ~1e-7 instead of 0 and, for grazing rays, the first root
// lands at t ~ 1e-4 > tmin — a phantom re-hit that makes a mirror sphere reflect into itself.  For the
// origin sphere the exact second root -2(b/2)/a is used instead: what the reference computes, without
// the cancellation.
RT_DEV float sphere_t_at(const float* __restrict__ im, const Ray<float>& r, bool is_origin) {
  float tm, half;
  const bool cross = sphere_cross(im, r, tm, half);
  if (is_origin) {
    const float t = 2.0f * tm;  // -2 (b/2) / a
    return (t > r.tmin && t < r.tmax) ? t : Num<float>::inf();
  }
  if (!cross) return Num<float>::inf();
  const float t1 = tm - half, t2 = tm + half;  // the first root inside (tmin, tmax), shapes.py:112-119
  if (t1 > r.tmin && t1 < r.tmax) return t1;
  if (t2 > r.tmin && t2 < r.tmax) return t2;
  return Num<float>::inf();
}

RT_DEV void resolve_candidates(const float* __restrict__ invm, int n_spheres, const int* cand, int nc,
                               const Ray<float>& r, float& best_t, int& best, int origin = -1) {
  if (nc <= RT_CAND_CAP) {
    for (int j = 0; j < nc; ++j) {
      const int i = cand[j];
      const float t = sphere_t_at(invm + 12 * (size_t)i, r, i == origin);
      if (t < best_t) { best_t = t; best = i; }
    }
  } else {  // a line through more than RT_CAND_CAP spheres: plain pass
    for (int i = 0; i < n_spheres; ++i) {
      const float t = sphere_t_at(invm + 12 * (size_t)i, r, i == origin);
      if (t < best_t) { best_t = t; best = i; }
    }
  }
}

RT_DEV bool sphere_blocks(const float* __restrict__ im, const Ray<float>& r) {
  float tm, half;
  if (!sphere_cross(im, r, tm, half)) return false;
  const float t1 = tm - half, t2 = tm + half;
  return (r.tmin < t1 && t1 < r.tmax) || (r.tmin < t2 && t2 < r.tmax);
}

RT_DEV bool any_candidate_blocks(const float* __restrict__ invm, int n_spheres, const int* cand, int nc,
                                 const Ray<float>& r) {
  if (nc <= RT_CAND_CAP) {
    for (int j = 0; j < nc; ++j)
      if (sphere_blocks(invm + 12 * (size_t)cand[j], r)) return true;
    return false;
  }
  for (int i = 0; i < n_spheres; ++i)
    if (sphere_blocks(invm + 12 * (size_t)i, r)) return true;
  return false;
}

// planes [0, n_planes) at `planes` (12 floats each; sorted index = n_spheres + k)
// (a ray that starts on a plane cannot meet it again: exact t = 0; the origin plane is skipped)
RT_DEV void scan_plane_block(const float* __restrict__ planes, int n_spheres, int n_planes,
                             const int32_t* __restrict__ orig, const Ray<float>& r, float& best_t, int& best,
                             int origin = -1) {
  for (int k = 0; k < n_planes; ++k) {
    const int i = n_spheres + k;
    if (i == origin) continue;
    const float t = plane_t<float>(planes + 12 * k, r);
    if (t < best_t) { best_t = t; best = i; }
    else if (t == best_t && best >= 0 && best < n_spheres) {
      if (plane_wins_tie(orig, i, best)) { best_t = t; best = i; }
    }
  }
}
RT_DEV bool any_plane_blocks(const float* __restrict__ planes, int n_planes, const Ray<float>& r) {
  for (int k = 0; k < n_planes; ++k)
    if (plane_t<float>(planes + 12 * k, r) < Num<float>::inf()) return true;
  return false;
}

// ---- where a kernel reads the scan data from (shared memory copy or global memory) ----------------
template <typename T> struct ScanSrc {  // generic: [n][12] inverse transforms
  const T* xf;
};
template <> struct ScanSrc<float> {     // fp32: packed pairs + plane records
  const float4* pairs;
  const float* planes;
};

template <typename T> RT_DEV ScanSrc<T> global_src(const SceneView<T>& sc) {
  ScanSrc<T> s;
  s.xf = sc.invm;
  return s;
}
template <> RT_DEV ScanSrc<float> global_src<float>(const SceneView<float>& sc) {
  ScanSrc<float> s;
  s.pairs = reinterpret_cast<const float4*>(sc.packed);
  s.planes = sc.packed + 24 * (size_t)sc.n_pairs;
  return s;
}

// World.ray_intersection's loop over ALL shapes (world.py:55-64): index of the winner, -1 = miss
// (`origin`, the shape a scattered ray starts on, is used by the fp32 path only — see resolve_candidates;
// the fp64 path evaluates every shape exactly like the reference does)
template <typename T>
RT_DEV void closest_all(const SceneView<T>& sc, const ScanSrc<T>& src, const Ray<T>& r, T& best_t, int& best, int origin = -1) {
  scan_closest<T>(src.xf, 0, sc.n_shapes, sc.n_spheres, sc.orig, r, best_t, best);
}
// all 32 lanes together (see sweep_pairs_split); `live` = this lane really has a ray
RT_DEV void closest_all_warp(const SceneView<float>& sc, const ScanSrc<float>& src, const Ray<float>& r, bool live,
                             float& best_t, int& best, int origin) {
  int cand[RT_CAND_CAP];
  int nc = 0;
  if (sc.n_pairs > 0) sweep_pairs_split(src.pairs, sc.n_pairs, r, sc.gate_a, sc.gate_t, cand, nc);
  if (live) {
    resolve_candidates(sc.invm, sc.n_spheres, cand, nc, r, best_t, best, origin);
    scan_plane_block(src.planes, sc.n_spheres, sc.n_shapes - sc.n_spheres, sc.orig, r, best_t, best, origin);
  }
}

template <bool UNROLL2>
RT_DEV void closest_all_f32(const SceneView<float>& sc, const ScanSrc<float>& src, const Ray<float>& r,
                            float& best_t, int& best, int origin = -1) {
  if (sc.n_pairs > 0) {
    int cand[RT_CAND_CAP];
    int nc = 0;
    const PackedRay pr = pack_ray(r, sc.gate_a, sc.gate_t);
    sweep_pairs<UNROLL2>(src.pairs, 0, 0, sc.n_pairs, pr, cand, nc);
    resolve_candidates(sc.invm, sc.n_spheres, cand, nc, r, best_t, best, origin);
  }
  scan_plane_block(src.planes, sc.n_spheres, sc.n_shapes - sc.n_spheres, sc.orig, r, best_t, best, origin);
}
template <>
RT_DEV void closest_all<float>(const SceneView<float>& sc, const ScanSrc<float>& src, const Ray<float>& r,
                               float& best_t, int& best, int origin) {
  closest_all_f32<true>(sc, src, r, best_t, best, origin);
}

// World.is_point_visible's loop (world.py:76-78): does any shape block the segment?
template <typename T> RT_DEV bool any_all(const SceneView<T>& sc, const ScanSrc<T>& src, const Ray<T>& r) {
  return scan_any<T>(src.xf, 0, sc.n_shapes, sc.n_spheres, r);
}
template <> RT_DEV bool any_all<float>(const SceneView<float>& sc, const ScanSrc<float>& src, const Ray<float>& r) {
  if (any_plane_blocks(src.planes, sc.n_shapes - sc.n_spheres, r)) return true;
  if (sc.n_pairs == 0) return false;
  int cand[RT_CAND_CAP];
  int nc = 0;
  const PackedRay pr = pack_ray(r, sc.gate_a, sc.gate_t);
  sweep_pairs(src.pairs, 0, 0, sc.n_pairs, pr, cand, nc);
  return any_candidate_blocks(sc.invm, sc.n_spheres, cand, nc, r);
}

// Hit record of the winning shape (shapes.py:123-131 / :176-189) + world.py:66-67, in three steps so
// that a caller can stop after the one it needs (the path tracer needs nothing but the emitted colour
// for a ray whose children would be cut, and no world frame when the surface does not scatter):
//   local_hit    ray and hit point in the shape's frame
//   local_uv     surface coordinates (shapes.py:36-42 sphere, :186-187 plane)
//   world_frame  world point and normal (shapes.py:45-54 / :176-183, normalised like world.py:66-67)
template <typename T> struct LocalHit {
  V3<T> hp, d;
};
template <typename T> RT_DEV LocalHit<T> local_hit(const T* im, const Ray<T>& r, T t) {
  LocalHit<T> L;
  V3<T> o = xf_point(im, r.o);
  L.d = xf_vec(im, r.d);
  L.hp = o + t * L.d;
  return L;
}
// the same two steps for the fp32 wavefront kernel, on transform rows already in registers
RT_DEV LocalHit<float> local_hit_rows(const Rows3& M, const Ray<float>& r, float t) {
  LocalHit<float> L;
  const V3<float> o = mk3<float>(fmaf(r.o.x, M.r0.x, fmaf(r.o.y, M.r0.y, fmaf(r.o.z, M.r0.z, M.r0.w))),
                                 fmaf(r.o.x, M.r1.x, fmaf(r.o.y, M.r1.y, fmaf(r.o.z, M.r1.z, M.r1.w))),
                                 fmaf(r.o.x, M.r2.x, fmaf(r.o.y, M.r2.y, fmaf(r.o.z, M.r2.z, M.r2.w))));
  L.d = mk3<float>(fmaf(r.d.x, M.r0.x, fmaf(r.d.y, M.r0.y, r.d.z * M.r0.z)),
                   fmaf(r.d.x, M.r1.x, fmaf(r.d.y, M.r1.y, r.d.z * M.r1.z)),
                   fmaf(r.d.x, M.r2.x, fmaf(r.d.y, M.r2.y, r.d.z * M.r2.z)));
  L.hp = o + t * L.d;
  return L;
}
RT_DEV void world_frame_rows(const Rows3& I, const Rows3& M, const LocalHit<float>& L, bool sphere, V3<float>& point, V3<float>& normal) {
  point = mk3<float>(fmaf(L.hp.x, M.r0.x, fmaf(L.hp.y, M.r0.y, fmaf(L.hp.z, M.r0.z, M.r0.w))),
                     fmaf(L.hp.x, M.r1.x, fmaf(L.hp.y, M.r1.y, fmaf(L.hp.z, M.r1.z, M.r1.w))),
                     fmaf(L.hp.x, M.r2.x, fmaf(L.hp.y, M.r2.y, fmaf(L.hp.z, M.r2.z, M.r2.w))));
  V3<float> n;
  if (sphere) n = (dot(L.hp, L.d) < 0.f) ? L.hp : -L.hp;  // shapes.py:45-54
  else n = mk3<float>(0.f, 0.f, (L.d.z < 0.f) ? 1.f : -1.f);
  n = mk3<float>(fmaf(n.x, I.r0.x, fmaf(n.y, I.r1.x, n.z * I.r2.x)),   // transpose of the inverse
                 fmaf(n.x, I.r0.y, fmaf(n.y, I.r1.y, n.z * I.r2.y)),
                 fmaf(n.x, I.r0.z, fmaf(n.y, I.r1.z, n.z * I.r2.z)));
  normal = normalize(n);
}
template <typename T> RT_DEV void local_uv(const LocalHit<T>& L, bool sphere, T& u_out, T& v_out) {
  if (sphere) {
    T u = Num<T>::atan2(L.hp.y, L.hp.x) / (T)(2.0 * 3.14159265358979323846);  // shapes.py:36-42
    u_out = (u >= (T)0) ? u : u + (T)1;
    T z = Num<T>::min((T)1, Num<T>::max((T)-1, L.hp.z));  // the reference would raise outside [-1,1]
    v_out = Num<T>::acos(z) / (T)3.14159265358979323846;
  } else {
    u_out = L.hp.x - Num<T>::floor(L.hp.x);
    v_out = L.hp.y - Num<T>::floor(L.hp.y);
  }
}
template <typename T>
RT_DEV void world_frame(const T* im, const T* mm, const LocalHit<T>& L, bool sphere, bool normalise, V3<T>& point, V3<T>& normal) {
  point = xf_point(mm, L.hp);
  V3<T> n;
  if (sphere) n = (dot(L.hp, L.d) < (T)0) ? L.hp : -L.hp;  // shapes.py:45-54
  else n = mk3<T>((T)0, (T)0, (L.d.z < (T)0) ? (T)1 : (T)-1);
  n = xf_normal(im, n);
  if (normalise) {
    if (Num<T>::is_f64) {  // Normal.normalize geometry.py:220-226
      T nn = Num<T>::sqrt(n.x * n.x + n.y * n.y + n.z * n.z);
      n = mk3<T>(n.x / nn, n.y / nn, n.z / nn);
    } else {
      n = normalize(n);
    }
  }
  normal = n;
}

template <typename T>
RT_DEV void finish_hit(const SceneView<T>& sc, const Ray<T>& r, T t, int idx, Hit<T>& h, bool normalise = true,
                       bool force_uv = false) {
  const T* im = sc.invm + 12 * (size_t)idx;
  const bool sphere = idx < sc.n_spheres;
  const LocalHit<T> L = local_hit<T>(im, r, t);
  h.idx = idx;
  h.t = t;
  h.u = h.v = (T)0;
  // a plane's (u, v) cost two floors; a sphere's atan2 / acos are skipped when no pigment reads them
  if (!sphere || force_uv || (sc.materials[sc.material[idx]].flags & MAT_USES_UV)) local_uv<T>(L, sphere, h.u, h.v);
  world_frame<T>(im, sc.m + 12 * (size_t)idx, L, sphere, normalise, h.point, h.normal);
}

// ---------------------------------------------------------------- pigments
template <typename T> RT_DEV V3<T> pig_c1(const DevPigment& p);
template <> RT_DEV V3<float> pig_c1<float>(const DevPigment& p) { return mk3<float>(p.c1[0], p.c1[1], p.c1[2]); }
template <> RT_DEV V3<double> pig_c1<double>(const DevPigment& p) { return mk3<double>(p.c1d[0], p.c1d[1], p.c1d[2]); }
template <typename T> RT_DEV V3<T> pig_c2(const DevPigment& p);
template <> RT_DEV V3<float> pig_c2<float>(const DevPigment& p) { return mk3<float>(p.c2[0], p.c2[1], p.c2[2]); }
template <> RT_DEV V3<double> pig_c2<double>(const DevPigment& p) { return mk3<double>(p.c2d[0], p.c2d[1], p.c2d[2]); }

template <typename T> RT_DEV V3<T> pig_texel(const DevPigment& p, int col, int row);
// out of line: image pigments are the rare case and the fetch must not be if-converted into the
// uniform / checkered paths
static __device__ __noinline__ float4 fetch_texel(cudaTextureObject_t tex, float x, float y) {
  return tex2D<float4>(tex, x, y);  // texture unit, nearest texel
}
template <> RT_DEV V3<float> pig_texel<float>(const DevPigment& p, int col, int row) {
  float4 t = fetch_texel(p.tex, col + 0.5f, row + 0.5f);
  return mk3<float>(t.x, t.y, t.z);
}
template <> RT_DEV V3<double> pig_texel<double>(const DevPigment& p, int col, int row) {
  const double* t = p.texels64 + 3 * ((size_t)row * p.tex_w + col);
  return mk3<double>(t[0], t[1], t[2]);
}

template <typename T> RT_DEV V3<T> pigment_color(const DevPigment* pigs, int idx, T u, T v) {
  const DevPigment& p = pigs[idx];
  if (p.kind == RT_PIGMENT_UNIFORM) return pig_c1<T>(p);  // materials.py:58
  if (p.kind == RT_PIGMENT_CHECKERED) {                   // materials.py:96-100
    long long iu = Num<T>::floor_ll(u * (T)p.steps);
    long long iv = Num<T>::floor_ll(v * (T)p.steps);
    return ((iu & 1) == (iv & 1)) ? pig_c1<T>(p) : pig_c2<T>(p);
  }
  int col = (int)(u * (T)p.tex_w);                        // materials.py:70-82
  int row = (int)(v * (T)p.tex_h);
  col = min(max(col, 0), p.tex_w - 1);
  row = min(max(row, 0), p.tex_h - 1);
  return pig_texel<T>(p, col, row);
}

// ---------------------------------------------------------------- BRDFs
template <typename T> RT_DEV T normalized_dot(V3<T> a, V3<T> b) {  // geometry.py:265-276
  return dot(normalize(a), normalize(b));
}
template <typename T> RT_DEV T clamped_acos(T x) {
  return Num<T>::acos(Num<T>::min((T)1, Num<T>::max((T)-1, x)));
}

// BRDF.eval: DiffuseBRDF materials.py:129-130, SpecularBRDF materials.py:164-173
template <typename T>
RT_DEV V3<T> brdf_eval(const SceneView<T>& sc, const DevMaterial& mat, V3<T> normal, V3<T> in_dir,
                       V3<T> out_dir, T u, T v) {
  V3<T> c = pigment_color<T>(sc.pigments, mat.brdf_pigment, u, v);
  if (mat.brdf_kind == RT_BRDF_DIFFUSE) return (T)(1.0 / 3.14159265358979323846) * c;
  T theta_in = clamped_acos(normalized_dot(normal, in_dir));
  T theta_out = clamped_acos(normalized_dot(normal, out_dir));
  if (Num<T>::abs(theta_in - theta_out) < (T)mat.threshold) return c;
  return mk3<T>((T)0, (T)0, (T)0);
}

// create_onb_from_z geometry.py:247-262 (Duff et al.)
template <typename T> RT_DEV void onb_from_z(V3<T> n, V3<T>& e1, V3<T>& e2) {
  T sign = (n.z > (T)0) ? (T)1 : (T)-1;
  T a = Num<T>::div((T)-1, sign + n.z);
  T b = n.x * n.y * a;
  e1 = mk3<T>((T)1 + sign * n.x * n.x * a, sign * b, -sign * n.x);
  e2 = mk3<T>(b, sign + n.y * n.y * a, -n.y);
}

// DiffuseBRDF.scatter_ray materials.py:132-152: cosine-weighted direction around `normal`
template <typename T> RT_DEV V3<T> diffuse_dir(V3<T> normal, T u1, T u2) {
  V3<T> e1, e2;
  onb_from_z(normal, e1, e2);
  T cos_theta = Num<T>::sqrt(u1), sin_theta = Num<T>::sqrt((T)1 - u1);
  T phi = (T)(2.0 * 3.14159265358979323846) * u2;
  T s, c;
  Num<T>::sincos(phi, &s, &c);
  return (cos_theta * (c * e1) + cos_theta * (s * e2)) + sin_theta * normal;
}

// SpecularBRDF.scatter_ray materials.py:175-196: mirror direction
template <typename T> RT_DEV V3<T> specular_dir(V3<T> incoming, V3<T> normal) {
  V3<T> rd = normalize(incoming);
  V3<T> n = normalize(normal);
  T dp = dot(n, rd);
  return rd - dp * ((T)2 * n);
}

// ---------------------------------------------------------------- camera + image tracer
// Always evaluated in fp64 and then rounded to T: the primary rays are the reference's own rays
// (camera.py:59-78,103-124 after imagetracer.py:56-58), whatever T the tracing uses.
struct DevCamera {
  int32_t kind, _pad;
  double dist, aspect;
  double m[12];
};

// Camera.fire_ray(u, v), camera.py:59-78 / :103-124
RT_DEV void camera_fire_f64(const DevCamera& cam, double u, double v, V3<double>& o, V3<double>& d) {
  double sy = __dmul_rn(__dsub_rn(1.0, __dmul_rn(2.0, u)), cam.aspect);
  double sz = __dsub_rn(__dmul_rn(2.0, v), 1.0);
  V3<double> lo, ld;
  if (cam.kind == RT_CAMERA_PERSPECTIVE) {
    lo = mk3<double>(-cam.dist, 0.0, 0.0);
    ld = mk3<double>(cam.dist, sy, sz);
  } else {
    lo = mk3<double>(-1.0, sy, sz);
    ld = mk3<double>(1.0, 0.0, 0.0);
  }
  const double* m = cam.m;
  // explicit round-to-nearest ops: no fused multiply-add even in the fp32 translation unit
#define RT_ROW3(v, r) __dadd_rn(__dadd_rn(__dmul_rn(v.x, m[r]), __dmul_rn(v.y, m[r + 1])), __dmul_rn(v.z, m[r + 2]))
  o = mk3<double>(__dadd_rn(RT_ROW3(lo, 0), m[3]), __dadd_rn(RT_ROW3(lo, 4), m[7]), __dadd_rn(RT_ROW3(lo, 8), m[11]));
  d = mk3<double>(RT_ROW3(ld, 0), RT_ROW3(ld, 4), RT_ROW3(ld, 8));
#undef RT_ROW3
}

// ImageTracer.fire_ray, imagetracer.py:48-58
RT_DEV void camera_ray_f64(const DevCamera& cam, int width, int height, int col, int row,
                           double u_pixel, double v_pixel, V3<double>& o, V3<double>& d) {
  double u = __ddiv_rn(__dadd_rn((double)col, u_pixel), (double)width);
  double v = __dsub_rn(1.0, __ddiv_rn(__dadd_rn((double)row, v_pixel), (double)height));
  camera_fire_f64(cam, u, v, o, d);
}

// jitter of imagetracer.py:88-93 from the two draws of this sample
RT_DEV void jitter_f64(Pcg& aa, int ic, int ir, int S, double& u_pixel, double& v_pixel) {
  double r1 = pcg_random_float<double>(aa);
  double r2 = pcg_random_float<double>(aa);
  u_pixel = __ddiv_rn(__dadd_rn((double)ic, r1), (double)S);
  v_pixel = __ddiv_rn(__dadd_rn((double)ir, r2), (double)S);
}
