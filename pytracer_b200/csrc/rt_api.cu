// rt_api.cu — host side of the C-ABI declared in include/rt_api.h.
//
// Owns device memory (scene tables in fp32 and fp64, textures, scratch images, counters), builds
// the LCG jump table of the jitter stream, picks kernel / precision and launches on the caller's
// stream.  There is no CPU fallback anywhere: without a CUDA device every entry point fails with
// RT_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "rt_launch.h"
#include "rt_bvh.h"

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(RT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// Per-device scratch shared by every scene of the process (one caller thread, see rt_api.h): counters,
// timing events and the staging buffers of the host-buffer entry points.  Created on first use and kept
// for the life of the process, so that creating / destroying a scene costs one allocation and one copy.
struct Workspace {
  unsigned long long* counters = nullptr;       // device, CNT_SLOTS
  unsigned long long* counters_host = nullptr;  // pinned
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, t0 = nullptr, t1 = nullptr;
  uint64_t* replay = nullptr;
  size_t replay_cap = 0;
  void* image = nullptr;  // scratch image for the host-buffer entry point
  size_t image_cap = 0;
  int32_t* hit = nullptr;
  size_t hit_cap = 0;
  void* probe_buf = nullptr;
  size_t probe_cap = 0;
  int sm_count = 0;
  // tone mapping (rt_tonemap.cu): per-block partial sums, completion counter, result; LDR staging
  double* tm_partials = nullptr;
  unsigned int* tm_done = nullptr;
  double* tm_sum = nullptr;
  double* tm_sum_host = nullptr;  // pinned
  void* ldr = nullptr;
  size_t ldr_cap = 0;
  void* hdr_out = nullptr;
  size_t hdr_out_cap = 0;
  void* co = nullptr;  // per-(origin, sphere) gate records of the hybrid resolve kernel
  size_t co_cap = 0;
  void* adaptive = nullptr;  // rt_render_adaptive: per-pixel sums, pass outputs, pixel lists
  size_t adaptive_cap = 0;
  int32_t* count_host = nullptr;  // pinned: the length of the next pass's pixel list
};

struct rt_scene {
  int device = 0, sm_count = 0;
  int n_shapes = 0, n_spheres = 0, n_materials = 0, n_pigments = 0, n_lights = 0;
  void* arena = nullptr;  // ONE device allocation holding every table below
  float *invm32 = nullptr, *m32 = nullptr, *packed32 = nullptr;
  int n_pairs = 0;
  float gate_a = 0.f, gate_t = 0.f;  // slack of the fp32 sweep's gate (rt_device.cuh pack_ray)
  double *invm64 = nullptr, *m64 = nullptr;
  int32_t *orig = nullptr, *material = nullptr;
  DevMaterial* materials = nullptr;
  DevPigment* pigments = nullptr;
  DevLight* lights = nullptr;
  double* texels64 = nullptr;
  // host mirrors of the transform tables (sorted order) for rt_scene_update_transforms
  std::vector<float> h_invm32, h_m32, h_packed;
  std::vector<double> h_invm64, h_m64;
  std::vector<int> sorted_of_orig;  // World.shapes index -> sorted index
  // sphere hierarchy (RT_ACCEL_BVH), built on first use and again after a transform update
  void* bvh_nodes = nullptr;
  int32_t* bvh_prims = nullptr;
  bool bvh_valid = false;
  int bvh_n_nodes = 0, bvh_n_prims = 0, bvh_depth = 0;
  std::vector<cudaArray_t> arrays;
  std::vector<cudaTextureObject_t> textures;
  Workspace* ws = nullptr;
  LaunchInfo last_info = {0, 0};
  int last_precision = 0;
  bool pending = false;
};

static void set_gate_constants(rt_scene* s);

static int get_workspace(int device, Workspace** out) {
  static Workspace* table[64] = {nullptr};
  if (device < 0 || device >= 64) return fail(RT_ERR_INVALID, "device index %d", device);
  if (!table[device]) {
    Workspace* w = new Workspace();
    // (cudaGetDeviceProperties takes tens of milliseconds; one attribute query, once per device)
    cudaError_t e = cudaDeviceGetAttribute(&w->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc((void**)&w->counters, CNT_SLOTS * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMallocHost((void**)&w->counters_host, CNT_SLOTS * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaEventCreate(&w->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&w->ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&w->t0);
    if (e == cudaSuccess) e = cudaEventCreate(&w->t1);
    if (e != cudaSuccess) { delete w; return fail(RT_ERR_CUDA, "workspace: %s", cudaGetErrorString(e)); }
    table[device] = w;
  }
  *out = table[device];
  return RT_OK;
}

extern "C" int rt_api_version(void) { return RT_API_VERSION; }

extern "C" const char* rt_last_error(void) { return g_err; }

extern "C" int rt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" int rt_set_device(int device) {
  if (rt_device_count() <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU path");
  CU(cudaSetDevice(device));
  return RT_OK;
}

template <typename T> static SceneView<T> view_of(const rt_scene* s);
template <> SceneView<float> view_of<float>(const rt_scene* s) {
  SceneView<float> v;
  v.invm = s->invm32; v.m = s->m32; v.orig = s->orig; v.material = s->material;
  v.materials = s->materials; v.pigments = s->pigments; v.lights = s->lights;
  v.n_shapes = s->n_shapes; v.n_spheres = s->n_spheres; v.n_lights = s->n_lights;
  v.packed = s->packed32; v.n_pairs = s->n_pairs; v.gate_a = s->gate_a;
  v.n_materials = s->n_materials; v.n_pigments = s->n_pigments;
  v.bvh_nodes = (const float4*)s->bvh_nodes; v.bvh_prims = s->bvh_prims; v.accel = 0; v.gate_t = s->gate_t;
  return v;
}
template <> SceneView<double> view_of<double>(const rt_scene* s) {
  SceneView<double> v;
  v.invm = s->invm64; v.m = s->m64; v.orig = s->orig; v.material = s->material;
  v.materials = s->materials; v.pigments = s->pigments; v.lights = s->lights;
  v.n_shapes = s->n_shapes; v.n_spheres = s->n_spheres; v.n_lights = s->n_lights;
  v.packed = nullptr; v.n_pairs = 0; v.gate_a = 0.f;
  v.n_materials = s->n_materials; v.n_pigments = s->n_pigments;
  v.bvh_nodes = (const float4*)s->bvh_nodes; v.bvh_prims = s->bvh_prims; v.accel = 0; v.gate_t = 0.f;
  return v;
}

// Host-side staging of the scene arena: tables are appended 256-byte aligned, uploaded with one copy.
struct Arena {
  std::vector<unsigned char> host;
  template <typename T> size_t add(const std::vector<T>& v) {
    size_t off = (host.size() + 255) / 256 * 256;
    host.resize(off + std::max<size_t>(v.size(), 1) * sizeof(T), 0);
    if (!v.empty()) memcpy(host.data() + off, v.data(), v.size() * sizeof(T));
    return off;
  }
};

extern "C" void rt_scene_destroy(rt_scene* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  for (auto t : s->textures) cudaDestroyTextureObject(t);
  for (auto a : s->arrays) cudaFreeArray(a);
  cudaFree(s->arena);
  cudaFree(s->bvh_nodes);
  cudaFree(s->bvh_prims);
  delete s;
}

extern "C" int rt_scene_create(const rt_scene_desc* d, rt_scene** out) {
  if (!d || !out) return fail(RT_ERR_INVALID, "rt_scene_create: null argument");
  if (rt_device_count() <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU path");
  if (d->n_shapes < 0 || d->n_materials < 0 || d->n_pigments < 0 || d->n_lights < 0)
    return fail(RT_ERR_INVALID, "rt_scene_create: negative count");
  rt_scene* s = new rt_scene();
  *out = nullptr;
  cudaGetDevice(&s->device);
  s->n_shapes = d->n_shapes; s->n_materials = d->n_materials; s->n_pigments = d->n_pigments; s->n_lights = d->n_lights;

  // ---- shapes, sorted spheres first / planes after, World.shapes order kept inside each group
  std::vector<int> order;
  for (int pass = 0; pass < 2; ++pass)
    for (int i = 0; i < d->n_shapes; ++i) {
      int k = d->shape_kind[i];
      if (k != RT_SHAPE_SPHERE && k != RT_SHAPE_PLANE) { delete s; return fail(RT_ERR_INVALID, "shape %d: unknown kind %d", i, k); }
      if ((pass == 0) == (k == RT_SHAPE_SPHERE)) order.push_back(i);
    }
  std::vector<float> invm32, m32;
  std::vector<double> invm64, m64;
  std::vector<int32_t> orig, mat;
  for (int i : order) {
    if (d->shape_kind[i] == RT_SHAPE_SPHERE) s->n_spheres++;
    int mi = d->shape_material[i];
    if (mi < 0 || mi >= d->n_materials) { delete s; return fail(RT_ERR_INVALID, "shape %d: material index %d out of range", i, mi); }
    orig.push_back(i);
    mat.push_back(mi);
    for (int k = 0; k < 12; ++k) {
      double a = d->shape_invm[12 * (size_t)i + k], b = d->shape_m[12 * (size_t)i + k];
      invm64.push_back(a); m64.push_back(b);
      invm32.push_back((float)a); m32.push_back((float)b);
    }
  }
  int rc;
  if ((rc = get_workspace(s->device, &s->ws)) != RT_OK) { delete s; return rc; }
  s->sm_count = s->ws->sm_count;
  Arena arena;
  std::vector<std::pair<void**, size_t>> fixups;  // (pointer field, offset in the arena)
#define UP(field, vec) fixups.push_back({(void**)&s->field, arena.add(vec)});
  UP(invm32, invm32) UP(m32, m32) UP(invm64, invm64) UP(m64, m64) UP(orig, orig) UP(material, mat)
  // fp32 scan array: sphere pairs element-interleaved (operands of the packed FFMA2 sweep), odd count
  // padded with an all-zero record (never crossed), then the plane records
  // an even pair count for real scenes (the warp sweep splits the list between half-warps); tiny scenes
  // (demo.txt: one sphere) are not padded — every pair costs 30 FFMA2 per ray
  s->n_pairs = s->n_spheres > 8 ? ((s->n_spheres + 3) / 4) * 2 : (s->n_spheres + 1) / 2;
  std::vector<float> packed((size_t)s->n_pairs * 24 + (size_t)(s->n_shapes - s->n_spheres) * 12, 0.0f);
  for (int i = 0; i < s->n_spheres; ++i)
    for (int k = 0; k < 12; ++k) packed[(size_t)(i / 2) * 24 + 2 * k + (i & 1)] = invm32[12 * (size_t)i + k];
  for (int i = s->n_spheres; i < s->n_shapes; ++i)
    for (int k = 0; k < 12; ++k) packed[(size_t)s->n_pairs * 24 + 12 * (size_t)(i - s->n_spheres) + k] = invm32[12 * (size_t)i + k];
  UP(packed32, packed)
  s->sorted_of_orig.assign(d->n_shapes, 0);
  for (int j = 0; j < d->n_shapes; ++j) s->sorted_of_orig[orig[j]] = j;
  s->h_invm32 = invm32; s->h_m32 = m32; s->h_invm64 = invm64; s->h_m64 = m64; s->h_packed = packed;
  set_gate_constants(s);

  // ---- textures: fp64 copy for the fp64 path, float4 CUDA arrays behind texture objects for fp32
  std::vector<double> tex64;
  if (d->n_texels > 0) tex64.assign(d->texels, d->texels + 3 * (size_t)d->n_texels);
  const size_t tex64_off = arena.add(tex64);
  fixups.push_back({(void**)&s->texels64, tex64_off});
  std::vector<DevPigment> pigs(d->n_pigments);
  for (int i = 0; i < d->n_pigments; ++i) {
    const rt_pigment& p = d->pigments[i];
    DevPigment& q = pigs[i];
    memset(&q, 0, sizeof(q));
    q.kind = p.kind; q.steps = p.num_of_steps; q.tex_w = p.tex_width; q.tex_h = p.tex_height;
    for (int k = 0; k < 3; ++k) {
      q.c1d[k] = p.color1[k]; q.c2d[k] = p.color2[k];
      q.c1[k] = (float)p.color1[k]; q.c2[k] = (float)p.color2[k];
    }
    if (p.kind == RT_PIGMENT_IMAGE) {
      if (p.tex_width <= 0 || p.tex_height <= 0 || p.tex_offset < 0 ||
          p.tex_offset + (int64_t)p.tex_width * p.tex_height > d->n_texels) {
        rt_scene_destroy(s);
        return fail(RT_ERR_INVALID, "pigment %d: texture window outside the texel buffer", i);
      }
      q.texels64 = reinterpret_cast<const double*>(3 * (size_t)p.tex_offset * sizeof(double));  // + arena base, patched below
      std::vector<float4> texels((size_t)p.tex_width * p.tex_height);
      const double* src = d->texels + 3 * (size_t)p.tex_offset;
      for (size_t t = 0; t < texels.size(); ++t)
        texels[t] = make_float4((float)src[3 * t], (float)src[3 * t + 1], (float)src[3 * t + 2], 0.f);
      cudaChannelFormatDesc fmt = cudaCreateChannelDesc<float4>();
      cudaArray_t arr = nullptr;
      cudaError_t e = cudaMallocArray(&arr, &fmt, p.tex_width, p.tex_height);
      if (e == cudaSuccess) {
        s->arrays.push_back(arr);
        e = cudaMemcpy2DToArray(arr, 0, 0, texels.data(), p.tex_width * sizeof(float4), p.tex_width * sizeof(float4),
                                p.tex_height, cudaMemcpyHostToDevice);
      }
      cudaTextureObject_t tex = 0;
      if (e == cudaSuccess) {
        cudaResourceDesc res;
        memset(&res, 0, sizeof(res));
        res.resType = cudaResourceTypeArray;
        res.res.array.array = arr;
        cudaTextureDesc td;
        memset(&td, 0, sizeof(td));
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        e = cudaCreateTextureObject(&tex, &res, &td, nullptr);
        if (e == cudaSuccess) s->textures.push_back(tex);
      }
      if (e != cudaSuccess) {
        rt_scene_destroy(s);
        return fail(RT_ERR_CUDA, "texture for pigment %d: %s", i, cudaGetErrorString(e));
      }
      q.tex = tex;
    } else if (p.kind != RT_PIGMENT_UNIFORM && p.kind != RT_PIGMENT_CHECKERED) {
      rt_scene_destroy(s);
      return fail(RT_ERR_INVALID, "pigment %d: unknown kind %d", i, p.kind);
    }
  }
  // materials and lights first, pigments last: their fp64 texel pointers need the arena's device address
  std::vector<DevMaterial> mats(d->n_materials);
  for (int i = 0; i < d->n_materials; ++i) {
    const rt_material& m = d->materials[i];
    if (m.brdf_pigment < 0 || m.brdf_pigment >= d->n_pigments || m.emitted_pigment < 0 || m.emitted_pigment >= d->n_pigments ||
        (m.brdf_kind != RT_BRDF_DIFFUSE && m.brdf_kind != RT_BRDF_SPECULAR)) {
      rt_scene_destroy(s);
      return fail(RT_ERR_INVALID, "material %d: bad BRDF kind or pigment index", i);
    }
    mats[i].brdf_kind = m.brdf_kind; mats[i].brdf_pigment = m.brdf_pigment; mats[i].emitted_pigment = m.emitted_pigment;
    const rt_pigment& pb = d->pigments[m.brdf_pigment];
    const rt_pigment& pe = d->pigments[m.emitted_pigment];
    int flags = 0;
    if (pb.kind != RT_PIGMENT_UNIFORM) flags |= MAT_UV_BRDF;
    if (pe.kind != RT_PIGMENT_UNIFORM) flags |= MAT_UV_EMIT;
    // (the float casts are what the fp32 kernels see; a colour that only rounds to zero in fp32 is
    // not "black" for the fp64 kernels, which do not read these two flags)
    if (pe.kind == RT_PIGMENT_UNIFORM && pe.color1[0] == 0.0 && pe.color1[1] == 0.0 && pe.color1[2] == 0.0) flags |= MAT_EMIT_BLACK;
    if (pb.kind == RT_PIGMENT_UNIFORM && !(std::max(std::max(pb.color1[0], pb.color1[1]), pb.color1[2]) > 0.0)) flags |= MAT_NO_SCATTER;
    mats[i].flags = flags;
    mats[i].threshold = m.threshold_angle_rad;
  }
  UP(materials, mats)
  std::vector<DevLight> lights(d->n_lights);
  for (int i = 0; i < d->n_lights; ++i) {
    for (int k = 0; k < 3; ++k) { lights[i].pos[k] = d->lights[i].position[k]; lights[i].color[k] = d->lights[i].color[k]; }
    lights[i].radius = d->lights[i].linear_radius;
  }
  UP(lights, lights)
  const size_t pig_off = arena.add(pigs);
  fixups.push_back({(void**)&s->pigments, pig_off});
#undef UP
  cudaError_t e = cudaMalloc(&s->arena, arena.host.size());
  if (e != cudaSuccess) { rt_scene_destroy(s); return fail(RT_ERR_CUDA, "scene arena (%zu bytes): %s", arena.host.size(), cudaGetErrorString(e)); }
  for (auto& f : fixups) *f.first = (unsigned char*)s->arena + f.second;
  DevPigment* staged = reinterpret_cast<DevPigment*>(arena.host.data() + pig_off);
  for (int i = 0; i < d->n_pigments; ++i)
    if (staged[i].kind == RT_PIGMENT_IMAGE)
      staged[i].texels64 = reinterpret_cast<const double*>((unsigned char*)s->texels64 + (size_t)staged[i].texels64);
  e = cudaMemcpy(s->arena, arena.host.data(), arena.host.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { rt_scene_destroy(s); return fail(RT_ERR_CUDA, "scene upload: %s", cudaGetErrorString(e)); }
  *out = s;
  return RT_OK;
}

// Constants of the fp32 sweep's gate (rt_device.cuh pack_ray): sqrt(8 u) times the largest Frobenius norm of
// a sphere's inverse 3x3 block and the largest norm of its translation column.
static void set_gate_constants(rt_scene* s) {
  double a_max = 0.0, t_max = 0.0;
  for (int i = 0; i < s->n_spheres; ++i) {
    const double* m = s->h_invm64.data() + 12 * (size_t)i;
    double f = 0.0, t = 0.0;
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) f += m[4 * r + c] * m[4 * r + c];
      t += m[4 * r + 3] * m[4 * r + 3];
    }
    a_max = std::max(a_max, std::sqrt(f));
    t_max = std::max(t_max, std::sqrt(t));
  }
  const double k = std::sqrt(8.0 * 5.9604644775390625e-08);
  s->gate_a = std::isfinite(a_max) ? (float)(k * a_max) : 0.f;
  s->gate_t = std::isfinite(t_max) ? (float)(k * t_max) : 0.f;
}

// Animation (SURVEY §8f-4; the reference re-parses the scene per frame with `-d clock:VALUE`,
// scene_file.py:654-675 / main.py:122-128): only Transformation.m / .invm of some shapes change between
// frames, so the resident scene is patched in place — 336 B per shape over five tables — instead of
// being rebuilt.  Ordered on `stream` after the renders already enqueued there.
extern "C" int rt_scene_update_transforms(rt_scene* s, int32_t first, int32_t n, const double* m, const double* invm, void* stream) {
  if (!s || !m || !invm) return fail(RT_ERR_INVALID, "rt_scene_update_transforms: null argument");
  if (first < 0 || n < 0 || first + n > s->n_shapes) return fail(RT_ERR_INVALID, "shapes [%d, %d) outside the scene's %d shapes", first, first + n, s->n_shapes);
  if (n == 0) return RT_OK;
  CU(cudaSetDevice(s->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int n_planes_base = s->n_pairs * 24;
  for (int i = 0; i < n; ++i) {
    const int j = s->sorted_of_orig[first + i];
    for (int k = 0; k < 12; ++k) {
      const double a = invm[12 * (size_t)i + k], b = m[12 * (size_t)i + k];
      s->h_invm64[12 * (size_t)j + k] = a; s->h_m64[12 * (size_t)j + k] = b;
      s->h_invm32[12 * (size_t)j + k] = (float)a; s->h_m32[12 * (size_t)j + k] = (float)b;
      if (j < s->n_spheres) s->h_packed[(size_t)(j / 2) * 24 + 2 * k + (j & 1)] = (float)a;
      else s->h_packed[(size_t)n_planes_base + 12 * (size_t)(j - s->n_spheres) + k] = (float)a;
    }
  }
  CU(cudaMemcpyAsync(s->invm32, s->h_invm32.data(), s->h_invm32.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(s->m32, s->h_m32.data(), s->h_m32.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(s->invm64, s->h_invm64.data(), s->h_invm64.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(s->m64, s->h_m64.data(), s->h_m64.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(s->packed32, s->h_packed.data(), s->h_packed.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  set_gate_constants(s);
  s->bvh_valid = false;  // rebuilt by the next render that asks for it
  return RT_OK;
}

// x -> A_b x + C_b = (x -> MULT x + inc) composed 2^b times
static void build_jump_table(uint64_t inc, JumpTable* t) {
  uint64_t mult = RT_PCG_MULT, plus = inc;
  for (int b = 0; b < RT_JUMP_BITS; ++b) {
    t->mult[b] = mult;
    t->plus[b] = plus;
    plus = (mult + 1) * plus;
    mult = mult * mult;
  }
}

static int fill_args(const rt_scene* s, const rt_render_params* p, RenderArgs* a) {
  if (p->width <= 0 || p->height <= 0) return fail(RT_ERR_INVALID, "image size %dx%d", p->width, p->height);
  if (p->samples_per_side < 0) return fail(RT_ERR_INVALID, "samples_per_side %d", p->samples_per_side);
  if (p->algorithm < RT_ALGO_ONOFF || p->algorithm > RT_ALGO_POINTLIGHT) return fail(RT_ERR_INVALID, "algorithm %d", p->algorithm);
  if (p->camera.kind != RT_CAMERA_ORTHOGONAL && p->camera.kind != RT_CAMERA_PERSPECTIVE) return fail(RT_ERR_INVALID, "camera kind %d", p->camera.kind);
  if (p->part_mode != RT_PART_NONE && (p->part_count < 1 || p->part_rank < 0 || p->part_rank >= p->part_count))
    return fail(RT_ERR_INVALID, "partition rank %d of %d", p->part_rank, p->part_count);
  long long S2 = p->samples_per_side > 0 ? (long long)p->samples_per_side * p->samples_per_side : 1;
  if ((double)p->width * p->height * (double)S2 * 2.0 >= 17592186044416.0 /* 2^44 */) return fail(RT_ERR_INVALID, "too many samples for the jitter jump table");
  memset(a, 0, sizeof(*a));
  a->width = p->width; a->height = p->height; a->S = p->samples_per_side; a->algorithm = p->algorithm;
  a->cam.kind = p->camera.kind; a->cam.dist = p->camera.screen_distance; a->cam.aspect = p->camera.aspect_ratio;
  memcpy(a->cam.m, p->camera.m, sizeof(a->cam.m));
  for (int k = 0; k < 3; ++k) { a->background[k] = p->background[k]; a->onoff[k] = p->onoff_color[k]; a->ambient[k] = p->ambient[k]; }
  a->num_of_rays = p->num_of_rays; a->max_depth = p->max_depth; a->rr_limit = p->rr_limit; a->rng_mode = p->rng_mode;
  a->aa_state = p->aa_state; a->aa_inc = p->aa_inc; a->pt_state = p->pt_state; a->pt_inc = p->pt_inc | 1ull;
  a->part_mode = p->part_count > 1 ? p->part_mode : RT_PART_NONE;
  a->part_rank = p->part_rank; a->part_count = p->part_count > 1 ? p->part_count : 1;
  a->out_f64 = p->out_f64 ? 1 : 0;
  a->hit_mode = p->hit_mode;
  if (p->rows_layout != RT_ROWS_FULL && p->rows_layout != RT_ROWS_COMPACT) return fail(RT_ERR_INVALID, "rows_layout %d", p->rows_layout);
  a->rows_compact = (a->part_mode == RT_PART_ROWS && p->rows_layout == RT_ROWS_COMPACT) ? 1 : 0;
  a->n_peers = 0;
  if (p->n_peer_images != 0) {
    if (p->n_peer_images < 0 || p->n_peer_images > RT_MAX_PEERS) return fail(RT_ERR_INVALID, "n_peer_images %d", p->n_peer_images);
    if (a->part_mode != RT_PART_ROWS || a->rows_compact || a->out_f64 || p->n_peer_images != a->part_count)
      return fail(RT_ERR_INVALID, "peer_images need RT_PART_ROWS, RT_ROWS_FULL, an fp32 image and one image per rank");
    for (int k = 0; k < p->n_peer_images; ++k) {
      if (!p->peer_images[k]) return fail(RT_ERR_INVALID, "peer_images[%d] is null", k);
      a->peer_out[k] = (float*)p->peer_images[k];
    }
    a->n_peers = p->n_peer_images;
  }
  a->counters = s->ws->counters;
  build_jump_table(p->aa_inc, &a->jump);
  return RT_OK;
}

// rows of the image this rank traces (RT_PART_ROWS: rank, rank + count, ...)
static long long owned_rows(const RenderArgs& a) {
  long long rows = a.height;
  if (a.part_mode == RT_PART_ROWS && a.part_count > 1) rows = (a.height - a.part_rank + a.part_count - 1) / a.part_count;
  return std::max(rows, 0ll);
}
// samples (Renderer.__call__ invocations) this rank's share of the image holds
static long long make_pixel_count(const RenderArgs& a) {
  long long S2 = a.S > 0 ? (long long)a.S * a.S : 1;
  long long rows = owned_rows(a), strata = S2;
  if (a.part_mode == RT_PART_SPP && a.part_count > 1) strata = a.part_rank < S2 ? (S2 - a.part_rank + a.part_count - 1) / a.part_count : 0;
  return std::max(rows, 0ll) * a.width * strata;
}

static int ensure(void** ptr, size_t* cap, size_t bytes) {
  if (*cap >= bytes && *ptr) return RT_OK;
  if (*ptr) cudaFree(*ptr);
  *ptr = nullptr; *cap = 0;
  CU(cudaMalloc(ptr, bytes));
  *cap = bytes;
  return RT_OK;
}

extern "C" int rt_bvh_build_host(const double* m, int32_t n_spheres, float* nodes_out, int32_t cap_nodes, int32_t* prims_out,
                                 int32_t* n_nodes, int32_t* depth) {
  if (!m || !nodes_out || !prims_out || !n_nodes || !depth || n_spheres < 0) return fail(RT_ERR_INVALID, "rt_bvh_build_host: bad argument");
  BvhBuild b = bvh_build(m, n_spheres);
  if ((int64_t)b.nodes.size() > cap_nodes) return fail(RT_ERR_INVALID, "rt_bvh_build_host: %zu nodes, room for %d", b.nodes.size(), cap_nodes);
  static_assert(sizeof(BvhHostNode) == 64, "node layout");
  if (!b.nodes.empty()) memcpy(nodes_out, b.nodes.data(), b.nodes.size() * sizeof(BvhHostNode));
  if (!b.prims.empty()) memcpy(prims_out, b.prims.data(), b.prims.size() * sizeof(int32_t));
  *n_nodes = (int32_t)b.nodes.size();
  *depth = b.max_depth;
  return RT_OK;
}

// Builds (host, rt_bvh.h) and uploads the sphere hierarchy of the scene's current transformations.
static int ensure_bvh(rt_scene* s, cudaStream_t st) {
  if (s->bvh_valid) return RT_OK;
  BvhBuild b = bvh_build(s->h_m64.data(), s->n_spheres);
  if (b.nodes.empty()) {  // no spheres: one node that is never read (the traversal returns first)
    b.nodes.push_back(BvhHostNode());
    b.prims.push_back(0);
  }
  if (b.max_depth + 2 > 48) return fail(RT_ERR_INVALID, "sphere hierarchy of depth %d exceeds the traversal stack", b.max_depth);
  CU(cudaStreamSynchronize(st));  // a render still reading the old tree must finish first
  cudaFree(s->bvh_nodes); cudaFree(s->bvh_prims);
  s->bvh_nodes = nullptr; s->bvh_prims = nullptr;
  CU(cudaMalloc(&s->bvh_nodes, b.nodes.size() * sizeof(BvhHostNode)));
  CU(cudaMalloc((void**)&s->bvh_prims, b.prims.size() * sizeof(int32_t)));
  CU(cudaMemcpy(s->bvh_nodes, b.nodes.data(), b.nodes.size() * sizeof(BvhHostNode), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(s->bvh_prims, b.prims.data(), b.prims.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  s->bvh_n_nodes = (int)b.nodes.size();
  s->bvh_n_prims = (int)b.prims.size();
  s->bvh_depth = b.max_depth;
  s->bvh_valid = true;
  return RT_OK;
}

extern "C" int rt_render_device(rt_scene* s, const rt_render_params* p, void* d_out_rgb, int32_t* d_out_hit, void* stream) {
  if (!s || !p || (!d_out_rgb && p->n_peer_images <= 0)) return fail(RT_ERR_INVALID, "rt_render_device: null argument");
  CU(cudaSetDevice(s->device));
  cudaStream_t st = (cudaStream_t)stream;
  RenderArgs a;
  int rc = fill_args(s, p, &a);
  if (rc != RT_OK) return rc;
  a.out_rgb = d_out_rgb;
  a.out_hit = d_out_hit;
  const bool pt = p->algorithm == RT_ALGO_PATHTRACING;
  // the hybrid path needs a common ray origin (perspective camera) and sweeps every sphere (no hierarchy)
  const bool hybrid_ok = !pt && p->camera.kind == RT_CAMERA_PERSPECTIVE && p->accel == RT_ACCEL_NONE;
  int precision = p->precision;
  if (precision == RT_PRECISION_AUTO) precision = pt ? RT_PRECISION_F32 : (hybrid_ok ? RT_PRECISION_HYBRID : RT_PRECISION_F64);
  if (precision == RT_PRECISION_HYBRID && !hybrid_ok)
    return fail(RT_ERR_INVALID, "RT_PRECISION_HYBRID needs a deterministic renderer, a perspective camera and RT_ACCEL_NONE");
  if (precision != RT_PRECISION_F32 && precision != RT_PRECISION_F64 && precision != RT_PRECISION_HYBRID)
    return fail(RT_ERR_INVALID, "precision %d", p->precision);
  int variant = p->variant;
  const bool auto_variant = variant == RT_VARIANT_AUTO;
  if (pt) {
    if (p->num_of_rays < 1) return fail(RT_ERR_INVALID, "num_of_rays %d", p->num_of_rays);
    if (variant == RT_VARIANT_AUTO)
      variant = (p->rng_mode == RT_RNG_REPLAY || precision == RT_PRECISION_F64) ? RT_VARIANT_MEGA : RT_VARIANT_WARP;
    if (variant == RT_VARIANT_WARP && (p->rng_mode == RT_RNG_REPLAY || precision == RT_PRECISION_F64))
      return fail(RT_ERR_INVALID, "the warp variant is fp32 with per-sample streams; replay / fp64 need the mega variant");
    if (p->rng_mode == RT_RNG_REPLAY) {
      if (!p->replay_states) return fail(RT_ERR_INVALID, "RT_RNG_REPLAY without replay_states");
      long long S2 = p->samples_per_side > 0 ? (long long)p->samples_per_side * p->samples_per_side : 1;
      size_t bytes = (size_t)p->width * p->height * S2 * sizeof(uint64_t);
      if ((rc = ensure((void**)&s->ws->replay, &s->ws->replay_cap, bytes)) != RT_OK) return rc;
      CU(cudaMemcpyAsync(s->ws->replay, p->replay_states, bytes, cudaMemcpyHostToDevice, st));
      a.replay = s->ws->replay;
    }
  }
  // pixels of the device image: the whole frame, or only the rows this rank owns (RT_ROWS_COMPACT)
  size_t px = (size_t)p->width * (a.rows_compact ? (size_t)owned_rows(a) : (size_t)p->height);
  if (a.n_peers > 0 && pt && p->max_depth < 0) return fail(RT_ERR_INVALID, "peer_images with max_depth < 0");
  CU(cudaMemsetAsync(s->ws->counters, 0, CNT_SLOTS * sizeof(unsigned long long), st));
  // rows this rank does not own stay zero, so that a sum over ranks is the image
  const bool partial_rows = a.part_mode == RT_PART_ROWS && !a.rows_compact && a.n_peers == 0;
  long long S2 = p->samples_per_side > 0 ? (long long)p->samples_per_side * p->samples_per_side : 1;
  const bool no_strata = a.part_mode == RT_PART_SPP && a.part_rank >= S2;
  // a pixel nobody traces: no shape (-1), or zero rays under RT_HIT_RAY_COUNT, so that the counts of the
  // ranks add up to those of the whole image
  const int no_hit = a.hit_mode == RT_HIT_RAY_COUNT ? 0 : 0xff;
  if (partial_rows || no_strata) {
    CU(cudaMemsetAsync(d_out_rgb, 0, px * 3 * (a.out_f64 ? sizeof(double) : sizeof(float)), st));
    if (d_out_hit) CU(cudaMemsetAsync(d_out_hit, no_hit, px * sizeof(int32_t), st));
  }
  if (p->accel != RT_ACCEL_NONE && p->accel != RT_ACCEL_BVH) return fail(RT_ERR_INVALID, "accel %d", p->accel);
  const int accel = (p->accel == RT_ACCEL_BVH && s->n_spheres > 0) ? RT_ACCEL_BVH : RT_ACCEL_NONE;
  if (accel == RT_ACCEL_BVH && (rc = ensure_bvh(s, st)) != RT_OK) return rc;
  SceneView<float> v32 = view_of<float>(s);
  SceneView<double> v64 = view_of<double>(s);
  v32.accel = v64.accel = accel;
  s->last_info = {0, 0};
  s->last_precision = precision;
  CU(cudaEventRecord(s->ws->ev0, st));
  cudaError_t e = cudaSuccess;
  const char* why = nullptr;
  if (pt && p->max_depth < 0) {
    // render.py:100-101: every primary ray already has depth 0 > max_depth, so each sample is BLACK and
    // no ray is traced — the image is zero whatever the scene
    long long n = (long long)make_pixel_count(a);
    unsigned long long samples = (unsigned long long)n;
    e = cudaMemsetAsync(d_out_rgb, 0, px * 3 * (a.out_f64 ? sizeof(double) : sizeof(float)), st);
    if (e == cudaSuccess && d_out_hit) e = cudaMemsetAsync(d_out_hit, no_hit, px * sizeof(int32_t), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s->ws->counters + CNT_SAMPLES, &samples, sizeof(samples), cudaMemcpyHostToDevice, st);
    s->last_info.variant = variant;
  } else if (!pt && precision == RT_PRECISION_HYBRID) {
    if ((rc = ensure(&s->ws->co, &s->ws->co_cap, resolve_hybrid_table_bytes(s->n_spheres, s->n_lights))) != RT_OK) return rc;
    e = launch_resolve_hybrid(v64, a, (float*)s->ws->co, st, &s->last_info);
  } else if (!pt) {
    e = precision == RT_PRECISION_F64 ? launch_resolve<double>(v64, a, st, &s->last_info)
                                      : launch_resolve<float>(v32, a, st, &s->last_info);
  } else if (variant == RT_VARIANT_MEGA) {
    e = precision == RT_PRECISION_F64 ? launch_pt_mega<double>(v64, a, st, &s->last_info)
                                      : launch_pt_mega<float>(v32, a, st, &s->last_info);
    if (e == cudaErrorInvalidValue) why = "max_depth > 64 with num_of_rays > 1 is not supported by the mega variant";
  } else {
    e = launch_pt_warp(v32, a, st, s->sm_count, &s->last_info, &why, s->bvh_n_nodes, s->bvh_n_prims, s->bvh_depth);
    if (e == cudaErrorInvalidValue && why && auto_variant) {
      // a configuration the wavefront kernel refuses (work stack deeper than shared memory holds):
      // AUTO falls back to the depth-first megakernel instead of failing
      cudaGetLastError();
      why = nullptr;
      e = launch_pt_mega<float>(v32, a, st, &s->last_info);
      if (e == cudaErrorInvalidValue) why = "max_depth > 64 with num_of_rays > 1 is supported by neither path-tracer kernel";
    }
  }
  if (e != cudaSuccess) return fail(why ? RT_ERR_INVALID : RT_ERR_CUDA, "render launch: %s", why ? why : cudaGetErrorString(e));
  CU(cudaEventRecord(s->ws->ev1, st));
  CU(cudaMemcpyAsync(s->ws->counters_host, s->ws->counters, CNT_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  s->pending = true;
  return RT_OK;
}

extern "C" int rt_render_finish(rt_scene* s, void* stream, rt_stats* stats) {
  if (!s) return fail(RT_ERR_INVALID, "rt_render_finish: null scene");
  CU(cudaSetDevice(s->device));
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    if (s->pending) {
      stats->rays_closest = s->ws->counters_host[CNT_CLOSEST];
      stats->rays_shadow = s->ws->counters_host[CNT_SHADOW];
      stats->samples = s->ws->counters_host[CNT_SAMPLES];
      stats->overflow = (int32_t)s->ws->counters_host[CNT_OVERFLOW];
      float ms = 0.f;
      CU(cudaEventElapsedTime(&ms, s->ws->ev0, s->ws->ev1));
      stats->kernel_ms = ms;
      stats->total_ms = ms;
      stats->variant_used = s->last_info.variant;
      stats->precision_used = s->last_precision;
      stats->n_launches = s->last_info.n_launches;
    }
  }
  bool ovf = s->pending && s->ws->counters_host[CNT_OVERFLOW] != 0;
  s->pending = false;
  if (ovf) return fail(RT_ERR_OVERFLOW, "a warp work stack overflowed; the image is invalid");
  return RT_OK;
}

// rt_render in two halves, so that rt_render_multi can have every device working before it waits for any:
// enqueue = launch into the workspace image + the copy of the image (or of this rank's rows) to the host.
static int render_enqueue(rt_scene* s, const rt_render_params* p, void* out_rgb, int32_t* out_hit) {
  CU(cudaSetDevice(s->device));
  if (p->width <= 0 || p->height <= 0) return fail(RT_ERR_INVALID, "image size %dx%d", p->width, p->height);
  if (p->n_peer_images != 0) return fail(RT_ERR_INVALID, "peer_images belong to rt_render_device");
  // RT_ROWS_COMPACT: the device image holds this rank's rows only; they are copied to their places in the
  // caller's full-size host image (which other ranks may be filling at the same time: shared page-locked memory)
  const bool compact = p->part_mode == RT_PART_ROWS && p->part_count > 1 && p->rows_layout == RT_ROWS_COMPACT;
  if (compact && (p->part_rank < 0 || p->part_rank >= p->part_count)) return fail(RT_ERR_INVALID, "partition rank %d of %d", p->part_rank, p->part_count);
  const size_t rows = compact ? (size_t)((p->height - p->part_rank + p->part_count - 1) / p->part_count) : (size_t)p->height;
  const size_t px = (size_t)p->width * rows;
  const size_t px_bytes = 3 * (p->out_f64 ? sizeof(double) : sizeof(float));
  const size_t bytes = px * px_bytes;
  int rc;
  if ((rc = ensure(&s->ws->image, &s->ws->image_cap, std::max<size_t>(bytes, 16))) != RT_OK) return rc;
  if (out_hit && (rc = ensure((void**)&s->ws->hit, &s->ws->hit_cap, std::max<size_t>(px * sizeof(int32_t), 16))) != RT_OK) return rc;
  CU(cudaEventRecord(s->ws->t0, 0));
  rc = rt_render_device(s, p, s->ws->image, out_hit ? s->ws->hit : nullptr, nullptr);
  if (rc != RT_OK) return rc;
  cudaError_t e = cudaSuccess;
  if (!compact) {
    e = cudaMemcpyAsync(out_rgb, s->ws->image, bytes, cudaMemcpyDeviceToHost, 0);
    if (e == cudaSuccess && out_hit) e = cudaMemcpyAsync(out_hit, s->ws->hit, px * sizeof(int32_t), cudaMemcpyDeviceToHost, 0);
  } else if (rows > 0) {
    const size_t row_bytes = (size_t)p->width * px_bytes, hit_row = (size_t)p->width * sizeof(int32_t);
    e = cudaMemcpy2DAsync((char*)out_rgb + (size_t)p->part_rank * row_bytes, (size_t)p->part_count * row_bytes, s->ws->image, row_bytes,
                          row_bytes, rows, cudaMemcpyDeviceToHost, 0);
    if (e == cudaSuccess && out_hit)
      e = cudaMemcpy2DAsync((char*)out_hit + (size_t)p->part_rank * hit_row, (size_t)p->part_count * hit_row, s->ws->hit, hit_row, hit_row,
                            rows, cudaMemcpyDeviceToHost, 0);
  }
  if (e == cudaSuccess) e = cudaEventRecord(s->ws->t1, 0);
  if (e != cudaSuccess) return fail(RT_ERR_CUDA, "image copy: %s", cudaGetErrorString(e));
  return RT_OK;
}

static int render_collect(rt_scene* s, rt_stats* stats) {
  int rc = rt_render_finish(s, nullptr, stats);
  if (rc == RT_OK && stats) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, s->ws->t0, s->ws->t1) == cudaSuccess) stats->total_ms = ms;
  }
  return rc;
}

extern "C" int rt_render(rt_scene* s, const rt_render_params* p, void* out_rgb, int32_t* out_hit, rt_stats* stats) {
  if (!s || !p || !out_rgb) return fail(RT_ERR_INVALID, "rt_render: null argument");
  int rc = render_enqueue(s, p, out_rgb, out_hit);
  if (rc == RT_OK) rc = render_collect(s, stats);
  return rc;
}

// One image over the devices of a node from ONE process and one call (SURVEY §8b/e): scenes[i] is the same
// World resident on device i; device i traces the rows i, i + n, ... (interleaved: the cost per row varies
// widely) with the kernel it would run alone and copies exactly those rows into the caller's image.  Every
// pixel is written by one device, so the image is bit-identical to the single-device image and no
// collective is needed; all devices are launched before any is waited for.
extern "C" int rt_render_multi(rt_scene* const* scenes, int32_t n_scenes, const rt_render_params* p, void* out_rgb,
                               int32_t* out_hit, rt_stats* stats) {
  if (!scenes || n_scenes < 1 || !p || !out_rgb) return fail(RT_ERR_INVALID, "rt_render_multi: null argument");
  if (n_scenes > RT_MAX_PEERS * 8) return fail(RT_ERR_INVALID, "rt_render_multi: %d scenes", n_scenes);
  for (int i = 0; i < n_scenes; ++i) {
    if (!scenes[i]) return fail(RT_ERR_INVALID, "rt_render_multi: scene %d is null", i);
    for (int j = 0; j < i; ++j)
      if (scenes[j]->device == scenes[i]->device) return fail(RT_ERR_INVALID, "rt_render_multi: scenes %d and %d live on the same device", j, i);
  }
  if (n_scenes == 1) return rt_render(scenes[0], p, out_rgb, out_hit, stats);
  if (p->part_mode != RT_PART_NONE) return fail(RT_ERR_INVALID, "rt_render_multi splits the image itself: part_mode must be RT_PART_NONE");
  if (p->rng_mode == RT_RNG_REPLAY) return fail(RT_ERR_INVALID, "rt_render_multi: replay is a single-device mode");
  int entry_device = 0;
  CU(cudaGetDevice(&entry_device));
  int rc = RT_OK, launched = 0;
  for (int i = 0; i < n_scenes && rc == RT_OK; ++i) {
    rt_render_params q = *p;
    q.part_mode = RT_PART_ROWS;
    q.part_rank = i;
    q.part_count = n_scenes;
    q.rows_layout = RT_ROWS_COMPACT;
    rc = render_enqueue(scenes[i], &q, out_rgb, out_hit);
    if (rc == RT_OK) launched = i + 1;
  }
  char first_error[sizeof(g_err)];
  if (rc != RT_OK) memcpy(first_error, g_err, sizeof(g_err));
  rt_stats total;
  memset(&total, 0, sizeof(total));
  for (int i = 0; i < launched; ++i) {  // every launched device is drained, also after an error
    rt_stats st;
    int r = render_collect(scenes[i], &st);
    if (r != RT_OK) {
      if (rc == RT_OK) { rc = r; memcpy(first_error, g_err, sizeof(g_err)); }
      continue;
    }
    total.rays_closest += st.rays_closest;
    total.rays_shadow += st.rays_shadow;
    total.samples += st.samples;
    total.overflow |= st.overflow;
    total.n_launches += st.n_launches;
    total.kernel_ms = std::max(total.kernel_ms, st.kernel_ms);
    total.total_ms = std::max(total.total_ms, st.total_ms);
    total.variant_used = st.variant_used;
    total.precision_used = st.precision_used;
  }
  cudaSetDevice(entry_device);
  if (rc != RT_OK) { memcpy(g_err, first_error, sizeof(g_err)); return rc; }
  if (stats) *stats = total;
  return RT_OK;
}

// x -> MULT x + inc applied `delta` times (PCG.advance on the host, pcg.py)
static uint64_t lcg_advance(uint64_t state, uint64_t inc, uint64_t delta) {
  uint64_t acc_mult = 1, acc_plus = 0, cur_mult = RT_PCG_MULT, cur_plus = inc;
  for (; delta; delta >>= 1) {
    if (delta & 1) { acc_mult *= cur_mult; acc_plus = acc_plus * cur_mult + cur_plus; }
    cur_plus = (cur_mult + 1) * cur_plus;
    cur_mult *= cur_mult;
  }
  return acc_mult * state + acc_plus;
}

// Path tracing with an error map and noise-targeted passes (rt_api.h).  Every per-pixel quantity stays on
// the device for the whole call: pass p runs the error-map path tracer over the current pixel list (pass 0:
// the image), rt_adaptive.cu folds its means and SE^2 into the per-pixel sums and writes the next list;
// the host reads one count per pass.
extern "C" int rt_render_adaptive(rt_scene* s, const rt_render_params* p, const rt_adaptive_params* ap, float* out_rgb, float* out_err,
                                  int32_t* out_samples, rt_adaptive_stats* stats) {
  if (!s || !p || !ap || !out_rgb) return fail(RT_ERR_INVALID, "rt_render_adaptive: null argument");
  if (p->algorithm != RT_ALGO_PATHTRACING) return fail(RT_ERR_INVALID, "rt_render_adaptive: path tracing only");
  if (p->samples_per_side < 2) return fail(RT_ERR_INVALID, "rt_render_adaptive: samples_per_side %d (the error map needs >= 2)", p->samples_per_side);
  if (p->variant != RT_VARIANT_AUTO && p->variant != RT_VARIANT_WARP) return fail(RT_ERR_INVALID, "rt_render_adaptive: the warp variant only");
  if (p->precision != RT_PRECISION_AUTO && p->precision != RT_PRECISION_F32) return fail(RT_ERR_INVALID, "rt_render_adaptive: fp32 only");
  if (p->part_mode != RT_PART_NONE || p->n_peer_images != 0 || p->out_f64 || p->rng_mode != RT_RNG_STREAMS)
    return fail(RT_ERR_INVALID, "rt_render_adaptive: one device, RT_PART_NONE, RT_RNG_STREAMS, an fp32 image and no peer images");
  if (p->num_of_rays < 1 || p->max_depth < 0) return fail(RT_ERR_INVALID, "rt_render_adaptive: num_of_rays %d, max_depth %d", p->num_of_rays, p->max_depth);
  if (ap->max_passes < 1 || !(ap->error_floor > 0.0) || std::isnan(ap->target_error))
    return fail(RT_ERR_INVALID, "rt_render_adaptive: max_passes %d, error_floor %g, target_error %g", ap->max_passes, ap->error_floor, ap->target_error);
  if (ap->estimator != RT_ERR_EST_BATCH && ap->estimator != RT_ERR_EST_PAIRED)
    return fail(RT_ERR_INVALID, "rt_render_adaptive: estimator %d", ap->estimator);
  if (ap->estimator == RT_ERR_EST_PAIRED && p->samples_per_side % 2)  // a stratum without a partner
    return fail(RT_ERR_INVALID, "rt_render_adaptive: the paired estimator needs an even samples_per_side (got %d)", p->samples_per_side);
  if ((long long)p->width * p->height >= (1ll << 31)) return fail(RT_ERR_INVALID, "rt_render_adaptive: image too large");
  CU(cudaSetDevice(s->device));
  RenderArgs a;
  int rc = fill_args(s, p, &a);
  if (rc != RT_OK) return rc;
  Workspace* ws = s->ws;
  const int n = p->width * p->height;
  const int S2 = p->samples_per_side * p->samples_per_side;
  const int max_passes = ap->target_error > 0.0 ? ap->max_passes : 1;
  if (p->accel != RT_ACCEL_NONE && p->accel != RT_ACCEL_BVH) return fail(RT_ERR_INVALID, "accel %d", p->accel);
  const int accel = (p->accel == RT_ACCEL_BVH && s->n_spheres > 0) ? RT_ACCEL_BVH : RT_ACCEL_NONE;
  cudaStream_t st = 0;
  if (accel == RT_ACCEL_BVH && (rc = ensure_bvh(s, st)) != RT_OK) return rc;
  SceneView<float> v32 = view_of<float>(s);
  v32.accel = accel;
  // device layout: pass mean / SE^2 per list entry, per-pixel sums and pass counts, two lists, flags, tile counts
  const size_t n3 = 3 * (size_t)n * sizeof(float), tiles = (size_t)n / 2048 + 2;
  auto al = [](size_t x) { return (x + 255) / 256 * 256; };
  const size_t o_em = 0, o_ev = o_em + al(n3), o_sm = o_ev + al(n3), o_sv = o_sm + al(n3), o_np = o_sv + al(n3);
  const size_t o_l0 = o_np + al((size_t)n * 4), o_l1 = o_l0 + al((size_t)n * 4), o_fl = o_l1 + al((size_t)n * 4);
  const size_t o_bc = o_fl + al((size_t)n), o_cnt = o_bc + al(tiles * 4), total = o_cnt + 256;
  if ((rc = ensure(&ws->adaptive, &ws->adaptive_cap, total)) != RT_OK) return rc;
  if (!ws->count_host) CU(cudaMallocHost((void**)&ws->count_host, sizeof(int32_t)));
  unsigned char* base = (unsigned char*)ws->adaptive;
  float *em = (float*)(base + o_em), *ev = (float*)(base + o_ev), *sm = (float*)(base + o_sm), *sv = (float*)(base + o_sv);
  int32_t* n_pass = (int32_t*)(base + o_np);
  int32_t* lists[2] = {(int32_t*)(base + o_l0), (int32_t*)(base + o_l1)};
  uint8_t* flags = base + o_fl;
  int32_t *block_counts = (int32_t*)(base + o_bc), *d_count = (int32_t*)(base + o_cnt);

  rt_adaptive_stats out;
  memset(&out, 0, sizeof(out));
  LaunchInfo info = {0, RT_VARIANT_WARP};
  CU(cudaEventRecord(ws->t0, st));
  CU(cudaMemsetAsync(ws->counters, 0, CNT_SLOTS * sizeof(unsigned long long), st));
  CU(cudaEventRecord(ws->ev0, st));
  const uint64_t draws_per_image = 2ull * (uint64_t)n * (uint64_t)S2;
  long long n_cur = n;
  int passes = 0;
  for (int pass = 0; pass < max_passes && n_cur > 0; ++pass) {
    // pass p = the (p+1)-th consecutive image: ImageTracer.pcg after p images, PathTracer.pcg after p random() calls
    a.aa_state = lcg_advance(p->aa_state, p->aa_inc, (uint64_t)pass * draws_per_image);
    a.pt_state = lcg_advance(p->pt_state, a.pt_inc, (uint64_t)pass);
    ErrArgs e;
    memset(&e, 0, sizeof(e));
    e.pix_list = pass == 0 ? nullptr : lists[pass & 1];
    e.n_list = n_cur;
    e.err_mean = em;
    e.err_var = ev;
    e.estimator = ap->estimator;
    CU(cudaMemsetAsync(ws->counters + CNT_TASK, 0, sizeof(unsigned long long), st));
    const char* why = nullptr;
    cudaError_t err = launch_pt_warp_err(v32, a, e, st, s->sm_count, &info, &why, s->bvh_n_nodes, s->bvh_n_prims, s->bvh_depth);
    if (err != cudaSuccess) return fail(why ? RT_ERR_INVALID : RT_ERR_CUDA, "rt_render_adaptive: %s", why ? why : cudaGetErrorString(err));
    err = launch_adaptive_combine(e, pass, max_passes, (float)ap->target_error, (float)ap->error_floor, sm, sv, n_pass, flags, block_counts,
                                  d_count, lists[(pass + 1) & 1], n, st, &info);
    if (err != cudaSuccess) return fail(RT_ERR_CUDA, "rt_render_adaptive: %s", cudaGetErrorString(err));
    if (pass < 16) out.pixels_in_pass[pass] = n_cur;
    passes = pass + 1;
    if (pass + 1 < max_passes) {  // the one host read of the pass: how many pixels the next pass traces
      CU(cudaMemcpyAsync(ws->count_host, d_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      n_cur = *ws->count_host;
    }
  }
  cudaError_t err = launch_adaptive_final(sm, sv, n_pass, S2, n, em, out_err ? ev : nullptr, out_samples ? lists[0] : nullptr, st, &info);
  if (err != cudaSuccess) return fail(RT_ERR_CUDA, "rt_render_adaptive: %s", cudaGetErrorString(err));
  CU(cudaEventRecord(ws->ev1, st));
  CU(cudaMemcpyAsync(out_rgb, em, n3, cudaMemcpyDeviceToHost, st));
  if (out_err) CU(cudaMemcpyAsync(out_err, ev, n3, cudaMemcpyDeviceToHost, st));
  if (out_samples) CU(cudaMemcpyAsync(out_samples, lists[0], (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(ws->counters_host, ws->counters, CNT_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CU(cudaEventRecord(ws->t1, st));
  CU(cudaStreamSynchronize(st));
  out.rays_closest = ws->counters_host[CNT_CLOSEST];
  out.rays_shadow = ws->counters_host[CNT_SHADOW];
  out.samples = ws->counters_host[CNT_SAMPLES];
  out.overflow = (int32_t)ws->counters_host[CNT_OVERFLOW];
  out.passes = passes;
  out.n_launches = info.n_launches;
  CU(cudaEventElapsedTime(&out.kernel_ms, ws->ev0, ws->ev1));
  CU(cudaEventElapsedTime(&out.total_ms, ws->t0, ws->t1));
  s->pending = false;
  if (stats) *stats = out;
  if (out.overflow) return fail(RT_ERR_OVERFLOW, "a warp work stack overflowed; the image is invalid");
  return RT_OK;
}

// ------------------------------------------------------------------------------------ probes
// Generic probe runner: packs `in` (and optional depth / pcg) into the scene's probe buffer, runs
// k_probe in the requested precision, copies the outputs back.  Blocking; default stream.
static int run_probe(rt_scene* s, int precision, const rt_render_params* p, int what, int n, int aux,
                     const void* in, size_t in_bytes, const int32_t* depth, uint64_t* pcg,
                     void* out, size_t out_bytes, int out_kind /*0 double,1 hits,2 flags,3 draws*/) {
  if (!s) return fail(RT_ERR_INVALID, "probe: null scene");
  CU(cudaSetDevice(s->device));
  RenderArgs a;
  rt_render_params dflt;
  if (!p) {
    memset(&dflt, 0, sizeof(dflt));
    dflt.width = dflt.height = 1;
    dflt.camera.kind = RT_CAMERA_PERSPECTIVE;
    dflt.camera.screen_distance = dflt.camera.aspect_ratio = 1.0;
    dflt.camera.m[0] = dflt.camera.m[5] = dflt.camera.m[10] = 1.0;
    dflt.num_of_rays = 1;
    p = &dflt;
  }
  int rc = fill_args(s, p, &a);
  if (rc != RT_OK) return rc;
  if (precision == RT_PRECISION_AUTO || precision == RT_PRECISION_HYBRID) precision = RT_PRECISION_F64;  // single items: plain fp64
  auto align = [](size_t x) { return (x + 255) / 256 * 256; };
  size_t off_in = 0, off_depth = align(in_bytes), off_pcg = off_depth + align(depth ? n * sizeof(int32_t) : 0);
  size_t off_out = off_pcg + 256, total = off_out + align(out_bytes);
  if ((rc = ensure(&s->ws->probe_buf, &s->ws->probe_cap, total)) != RT_OK) return rc;
  unsigned char* base = (unsigned char*)s->ws->probe_buf;
  if (in_bytes) CU(cudaMemcpy(base + off_in, in, in_bytes, cudaMemcpyHostToDevice));
  if (depth) CU(cudaMemcpy(base + off_depth, depth, n * sizeof(int32_t), cudaMemcpyHostToDevice));
  if (pcg) CU(cudaMemcpy(base + off_pcg, pcg, 2 * sizeof(uint64_t), cudaMemcpyHostToDevice));
  CU(cudaMemset(s->ws->counters, 0, CNT_SLOTS * sizeof(unsigned long long)));
  ProbeArgs pa;
  memset(&pa, 0, sizeof(pa));
  pa.what = what; pa.n = n; pa.aux = aux;
  pa.in = (const double*)(base + off_in);
  pa.depth = depth ? (const int32_t*)(base + off_depth) : nullptr;
  pa.pcg = (uint64_t*)(base + off_pcg);
  pa.out = (double*)(base + off_out);
  pa.hits = (rt_hit*)(base + off_out);
  pa.flags = (uint8_t*)(base + off_out);
  pa.draws = (uint32_t*)(base + off_out);
  (void)out_kind;
  cudaError_t e = precision == RT_PRECISION_F64 ? launch_probe<double>(view_of<double>(s), a, pa, 0)
                                                : launch_probe<float>(view_of<float>(s), a, pa, 0);
  if (e != cudaSuccess) return fail(RT_ERR_CUDA, "probe launch: %s", cudaGetErrorString(e));
  CU(cudaDeviceSynchronize());
  if (out_bytes) CU(cudaMemcpy(out, base + off_out, out_bytes, cudaMemcpyDeviceToHost));
  if (pcg) CU(cudaMemcpy(pcg, base + off_pcg, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return RT_OK;
}

extern "C" int rt_trace_rays(rt_scene* s, const rt_render_params* p, const double* rays, const int32_t* depth,
                             int32_t n, uint64_t* pcg_state_inc, double* out_rgb) {
  if (!p || !rays || !out_rgb || n < 0) return fail(RT_ERR_INVALID, "rt_trace_rays: bad argument");
  if (n == 0) return RT_OK;
  uint64_t local[2] = {p->pt_state, p->pt_inc};
  uint64_t* pcg = pcg_state_inc ? pcg_state_inc : local;
  int precision = p->precision == RT_PRECISION_AUTO ? RT_PRECISION_F64 : p->precision;
  if (p->algorithm == RT_ALGO_PATHTRACING && p->num_of_rays > 1 && p->max_depth > 64)
    return fail(RT_ERR_INVALID, "rt_trace_rays: max_depth > 64 with num_of_rays > 1");
  return run_probe(s, precision, p, PROBE_TRACE, n, 0, rays, (size_t)n * 8 * sizeof(double), depth, pcg, out_rgb,
                   (size_t)n * 3 * sizeof(double), 0);
}

extern "C" int rt_intersect(rt_scene* s, int32_t precision, int32_t normalize_normal, const double* rays, int32_t n, rt_hit* out) {
  if (!rays || !out || n < 0) return fail(RT_ERR_INVALID, "rt_intersect: bad argument");
  if (n == 0) return RT_OK;
  return run_probe(s, precision, nullptr, PROBE_INTERSECT, n, normalize_normal ? 1 : 0, rays, (size_t)n * 8 * sizeof(double), nullptr,
                   nullptr, out, (size_t)n * sizeof(rt_hit), 1);
}

extern "C" int rt_is_point_visible(rt_scene* s, int32_t precision, const double* pairs, int32_t n, uint8_t* out) {
  if (!pairs || !out || n < 0) return fail(RT_ERR_INVALID, "rt_is_point_visible: bad argument");
  if (n == 0) return RT_OK;
  return run_probe(s, precision, nullptr, PROBE_VISIBLE, n, 0, pairs, (size_t)n * 6 * sizeof(double), nullptr, nullptr, out, (size_t)n, 2);
}

extern "C" int rt_pigment_color(rt_scene* s, int32_t pigment, int32_t precision, const double* uv, int32_t n, double* out_rgb) {
  if (!s || !uv || !out_rgb || n < 0) return fail(RT_ERR_INVALID, "rt_pigment_color: bad argument");
  if (pigment < 0 || pigment >= s->n_pigments) return fail(RT_ERR_INVALID, "pigment index %d out of range", pigment);
  if (n == 0) return RT_OK;
  return run_probe(s, precision, nullptr, PROBE_PIGMENT, n, pigment, uv, (size_t)n * 2 * sizeof(double), nullptr, nullptr, out_rgb,
                   (size_t)n * 3 * sizeof(double), 0);
}

extern "C" int rt_scatter(rt_scene* s, int32_t material, int32_t precision, const double* in, int32_t n,
                          uint64_t* state_inc, double* out_rays) {
  if (!s || !in || !out_rays || !state_inc || n < 0) return fail(RT_ERR_INVALID, "rt_scatter: bad argument");
  if (material < 0 || material >= s->n_materials) return fail(RT_ERR_INVALID, "material index %d out of range", material);
  if (n == 0) return RT_OK;
  return run_probe(s, precision, nullptr, PROBE_SCATTER, n, material, in, (size_t)n * 9 * sizeof(double), nullptr, state_inc,
                   out_rays, (size_t)n * 8 * sizeof(double), 0);
}

// The scene-free probes run on a scratch empty scene.
static int with_empty_scene(rt_scene** out) {
  static thread_local rt_scene* empty = nullptr;
  if (!empty) {
    rt_scene_desc d;
    memset(&d, 0, sizeof(d));
    int rc = rt_scene_create(&d, &empty);
    if (rc != RT_OK) return rc;
  }
  *out = empty;
  return RT_OK;
}

extern "C" int rt_onb(int32_t precision, const double* normals, int32_t n, double* out) {
  if (!normals || !out || n < 0) return fail(RT_ERR_INVALID, "rt_onb: bad argument");
  rt_scene* s;
  int rc = with_empty_scene(&s);
  if (rc != RT_OK) return rc;
  if (n == 0) return RT_OK;
  return run_probe(s, precision, nullptr, PROBE_ONB, n, 0, normals, (size_t)n * 3 * sizeof(double), nullptr, nullptr, out,
                   (size_t)n * 9 * sizeof(double), 0);
}

extern "C" int rt_pcg_draw(uint64_t* state_inc, int32_t n, uint32_t* out) {
  if (!state_inc || !out || n < 0) return fail(RT_ERR_INVALID, "rt_pcg_draw: bad argument");
  rt_scene* s;
  int rc = with_empty_scene(&s);
  if (rc != RT_OK) return rc;
  if (n == 0) return RT_OK;
  return run_probe(s, RT_PRECISION_F32, nullptr, PROBE_PCG_DRAW, n, 0, nullptr, 0, nullptr, state_inc, out, (size_t)n * sizeof(uint32_t), 3);
}

extern "C" int rt_pcg_seed(uint64_t init_state, uint64_t init_seq, uint64_t* state_inc) {
  if (!state_inc) return fail(RT_ERR_INVALID, "rt_pcg_seed: bad argument");
  rt_scene* s;
  int rc = with_empty_scene(&s);
  if (rc != RT_OK) return rc;
  state_inc[0] = init_state;
  state_inc[1] = init_seq;
  return run_probe(s, RT_PRECISION_F32, nullptr, PROBE_PCG_SEED, 1, 0, nullptr, 0, nullptr, state_inc, nullptr, 0, 0);
}

extern "C" int rt_camera_rays(const rt_render_params* p, int32_t precision, double* out_rays) {
  if (!p || !out_rays) return fail(RT_ERR_INVALID, "rt_camera_rays: bad argument");
  rt_scene* s;
  int rc = with_empty_scene(&s);
  if (rc != RT_OK) return rc;
  long long S2 = p->samples_per_side > 0 ? (long long)p->samples_per_side * p->samples_per_side : 1;
  long long total = (long long)p->width * p->height * S2;
  if (total <= 0 || total > (1ll << 28)) return fail(RT_ERR_INVALID, "rt_camera_rays: %lld rays", total);
  return run_probe(s, precision, p, PROBE_CAMERA_RAYS, (int)total, 0, nullptr, 0, nullptr, nullptr, out_rays,
                   (size_t)total * 8 * sizeof(double), 0);
}

extern "C" int rt_camera_fire(const rt_camera* cam, int32_t precision, const double* uv, int32_t n, double* out_rays) {
  if (!cam || !uv || !out_rays || n < 0) return fail(RT_ERR_INVALID, "rt_camera_fire: bad argument");
  rt_scene* s;
  int rc = with_empty_scene(&s);
  if (rc != RT_OK) return rc;
  if (n == 0) return RT_OK;
  rt_render_params p;
  memset(&p, 0, sizeof(p));
  p.width = p.height = 1;
  p.camera = *cam;
  p.num_of_rays = 1;
  return run_probe(s, precision, &p, PROBE_CAMERA_UV, n, 0, uv, (size_t)n * 2 * sizeof(double), nullptr, nullptr, out_rays,
                   (size_t)n * 8 * sizeof(double), 0);
}

// FMA throughput probes (fp64 = 0: FFMA, 1: DFMA): 8 independent chains per thread, 2048 threads per SM
static int bench_fma(int fp64, int32_t iterations, double* tflops, float* ms_out) {
  if (rt_device_count() <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU path");
  if (iterations < 1) iterations = 1;
  int dev = 0, sms = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int blocks = sms * 8;
  void* out = nullptr;
  CU(cudaMalloc(&out, (size_t)blocks * 256 * sizeof(double)));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  auto launch = [&]() { return fp64 ? launch_dfma((double*)out, blocks, iterations, 0) : launch_ffma((float*)out, blocks, iterations, 0); };
  cudaError_t e = launch();  // warm-up
  if (e == cudaSuccess) e = cudaEventRecord(e0, 0);
  if (e == cudaSuccess) e = launch();
  if (e == cudaSuccess) e = cudaEventRecord(e1, 0);
  if (e == cudaSuccess) e = cudaEventSynchronize(e1);
  float ms = 0.f;
  if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
  cudaFree(out);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (e != cudaSuccess) return fail(RT_ERR_CUDA, "FMA probe: %s", cudaGetErrorString(e));
  double flops = (double)blocks * 256.0 * (double)iterations * 16.0 * 8.0 * 2.0;
  if (tflops) *tflops = flops / (ms * 1e-3) / 1e12;
  if (ms_out) *ms_out = ms;
  return RT_OK;
}
extern "C" int rt_bench_ffma(int32_t iterations, double* tflops, float* ms) { return bench_fma(0, iterations, tflops, ms); }
extern "C" int rt_bench_dfma(int32_t iterations, double* tflops, float* ms) { return bench_fma(1, iterations, tflops, ms); }

// ------------------------------------------------------------------------------------ tone mapping
static int tonemap_workspace(Workspace** out) {
  if (rt_device_count() <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU path");
  int device = 0;
  CU(cudaGetDevice(&device));
  Workspace* w = nullptr;
  int rc = get_workspace(device, &w);
  if (rc != RT_OK) return rc;
  if (!w->tm_partials) {
    CU(cudaMalloc((void**)&w->tm_partials, tonemap_max_blocks() * sizeof(double)));
    CU(cudaMalloc((void**)&w->tm_done, sizeof(unsigned int)));
    CU(cudaMemset(w->tm_done, 0, sizeof(unsigned int)));
    CU(cudaMalloc((void**)&w->tm_sum, sizeof(double)));
    CU(cudaMallocHost((void**)&w->tm_sum_host, sizeof(double)));
  }
  *out = w;
  return RT_OK;
}

// device image -> average luminosity (hdrimages.py:120-128); synchronises `st`
static int device_average_luminosity(Workspace* w, const float* d_rgb, int64_t n_pixels, double delta, cudaStream_t st, double* out) {
  cudaError_t e = launch_lum_sum(d_rgb, n_pixels, delta, w->tm_partials, w->tm_done, w->tm_sum, w->sm_count, st);
  if (e != cudaSuccess) return fail(RT_ERR_CUDA, "luminosity launch: %s", cudaGetErrorString(e));
  CU(cudaMemcpyAsync(w->tm_sum_host, w->tm_sum, sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  *out = pow(10.0, *w->tm_sum_host / (double)n_pixels);
  return RT_OK;
}

extern "C" int rt_average_luminosity(const float* rgb, int64_t n_pixels, double delta, int32_t on_device, void* stream, double* out) {
  if (!rgb || !out) return fail(RT_ERR_INVALID, "rt_average_luminosity: null argument");
  if (n_pixels <= 0) return fail(RT_ERR_INVALID, "rt_average_luminosity: empty image (the reference divides by len(pixels))");
  Workspace* w = nullptr;
  int rc = tonemap_workspace(&w);
  if (rc != RT_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const float* d_rgb = rgb;
  if (!on_device) {
    const size_t bytes = (size_t)n_pixels * 3 * sizeof(float);
    if ((rc = ensure(&w->image, &w->image_cap, bytes)) != RT_OK) return rc;
    CU(cudaMemcpyAsync(w->image, rgb, bytes, cudaMemcpyHostToDevice, st));
    d_rgb = (const float*)w->image;
  }
  return device_average_luminosity(w, d_rgb, n_pixels, delta, st, out);
}

extern "C" int rt_tone_map(const float* rgb, int64_t n_pixels, int32_t flags, double factor, double luminosity, double gamma,
                           int32_t on_device, void* stream, float* out_hdr, uint8_t* out_ldr, rt_tonemap_stats* stats) {
  if (!rgb) return fail(RT_ERR_INVALID, "rt_tone_map: null image");
  if (n_pixels <= 0) return fail(RT_ERR_INVALID, "rt_tone_map: empty image");
  if (!(gamma > 0.0)) return fail(RT_ERR_INVALID, "rt_tone_map: gamma %g", gamma);
  Workspace* w = nullptr;
  int rc = tonemap_workspace(&w);
  if (rc != RT_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t px3 = (size_t)n_pixels * 3;
  const float* d_rgb = rgb;
  float* d_hdr = out_hdr;
  unsigned char* d_ldr = out_ldr;
  CU(cudaEventRecord(w->t0, st));
  if (!on_device) {
    if ((rc = ensure(&w->image, &w->image_cap, px3 * sizeof(float))) != RT_OK) return rc;
    CU(cudaMemcpyAsync(w->image, rgb, px3 * sizeof(float), cudaMemcpyHostToDevice, st));
    d_rgb = (const float*)w->image;
    if (out_hdr) { if ((rc = ensure(&w->hdr_out, &w->hdr_out_cap, px3 * sizeof(float))) != RT_OK) return rc; d_hdr = (float*)w->hdr_out; }
    if (out_ldr) { if ((rc = ensure(&w->ldr, &w->ldr_cap, px3)) != RT_OK) return rc; d_ldr = (unsigned char*)w->ldr; }
  }
  int launches = 0;
  float lum_ms = 0.f, map_ms = 0.f;
  // hdrimages.py:136-137 `if not luminosity`: None and 0.0 both mean "use the image's own average"
  if ((flags & RT_TONE_NORMALIZE) && (luminosity == 0.0 || luminosity != luminosity)) {
    CU(cudaEventRecord(w->ev0, st));
    cudaError_t e = launch_lum_sum(d_rgb, n_pixels, 1e-10, w->tm_partials, w->tm_done, w->tm_sum, w->sm_count, st);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "luminosity launch: %s", cudaGetErrorString(e));
    CU(cudaEventRecord(w->ev1, st));
    CU(cudaMemcpyAsync(w->tm_sum_host, w->tm_sum, sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    luminosity = pow(10.0, *w->tm_sum_host / (double)n_pixels);
    CU(cudaEventElapsedTime(&lum_ms, w->ev0, w->ev1));
    ++launches;
  }
  if (d_hdr || d_ldr) {
    CU(cudaEventRecord(w->ev0, st));
    cudaError_t e = launch_tone_map(d_rgb, n_pixels, flags, factor / luminosity, gamma, d_hdr, d_ldr, w->sm_count, st);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "tone map launch: %s", cudaGetErrorString(e));
    CU(cudaEventRecord(w->ev1, st));
    ++launches;
    if (!on_device) {
      if (out_hdr) CU(cudaMemcpyAsync(out_hdr, d_hdr, px3 * sizeof(float), cudaMemcpyDeviceToHost, st));
      if (out_ldr) CU(cudaMemcpyAsync(out_ldr, d_ldr, px3, cudaMemcpyDeviceToHost, st));
    }
  }
  CU(cudaEventRecord(w->t1, st));
  CU(cudaStreamSynchronize(st));
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    if (d_hdr || d_ldr) CU(cudaEventElapsedTime(&map_ms, w->ev0, w->ev1));
    float total = 0.f;
    CU(cudaEventElapsedTime(&total, w->t0, w->t1));
    stats->luminosity = luminosity;
    stats->lum_ms = lum_ms; stats->map_ms = map_ms; stats->total_ms = total;
    stats->n_launches = launches;
  }
  return RT_OK;
}

extern "C" int rt_host_register(void* ptr, uint64_t bytes) {
  if (!ptr || bytes == 0) return fail(RT_ERR_INVALID, "rt_host_register: bad argument");
  if (rt_device_count() <= 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU path");
  cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable);  // page-locked for every device of the process
  if (e == cudaErrorHostMemoryAlreadyRegistered) {
    // fine only if it is this very range that is registered (same caller pinning twice); an overlapping
    // older registration of a recycled address would leave part of the range pageable
    cudaGetLastError();
    cudaError_t u = cudaHostUnregister(ptr);
    if (u == cudaSuccess) e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable);
    else cudaGetLastError();
  }
  if (e != cudaSuccess) return fail(RT_ERR_CUDA, "cudaHostRegister: %s", cudaGetErrorString(e));
  return RT_OK;
}

extern "C" int rt_host_unregister(void* ptr) {
  if (!ptr) return fail(RT_ERR_INVALID, "rt_host_unregister: bad argument");
  cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(RT_ERR_CUDA, "cudaHostUnregister: %s", cudaGetErrorString(e)); }
  return RT_OK;
}
