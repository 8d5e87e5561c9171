/*
 * rt_api.h — C-ABI of the B200 rendering hot path (libpytracer_b200.so).
 *
 * The reference (ziotom78/pytracer) is pure Python and has no FFI: the seam this
 * library plugs into is the duck-typed call
 *     ImageTracer.fire_all_rays(func)              src/pytracer/imagetracer.py:60-110
 * with `func` one of the Renderer callables         src/pytracer/render.py:26-193.
 * One rt_render() call replaces the whole descent fire_all_rays -> Camera.fire_ray ->
 * Renderer.__call__ -> World.ray_intersection -> Shape/BRDF/Pigment/PCG for every pixel.
 * INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions: plain C structs of fixed-width types; every function returns 0 on success
 * and a negative code on failure (text via rt_last_error(), thread-local); no exception
 * crosses the ABI; the caller owns every buffer it passes; matrices are row-major 3x4
 * affine blocks (the first three rows of the reference's 4x4 lists) in fp64 — the library
 * derives its own fp32 mirrors. Image buffers are [height][width][3], row 0 = TOP of the
 * image, exactly HdrImage.pixel_offset (src/pytracer/hdrimages.py:78-80).
 */
#ifndef PYTRACER_B200_RT_API_H
#define PYTRACER_B200_RT_API_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_API_VERSION 1

/* Shape.kind: Sphere shapes.py:88, Plane shapes.py:154 */
enum { RT_SHAPE_SPHERE = 0, RT_SHAPE_PLANE = 1 };
/* DiffuseBRDF materials.py:123, SpecularBRDF materials.py:155 */
enum { RT_BRDF_DIFFUSE = 0, RT_BRDF_SPECULAR = 1 };
/* UniformPigment materials.py:50, CheckeredPigment :85, ImagePigment :62 */
enum { RT_PIGMENT_UNIFORM = 0, RT_PIGMENT_CHECKERED = 1, RT_PIGMENT_IMAGE = 2 };
/* OrthogonalCamera camera.py:42, PerspectiveCamera camera.py:82 */
enum { RT_CAMERA_ORTHOGONAL = 0, RT_CAMERA_PERSPECTIVE = 1 };
/* main.py:73 RENDERERS, in the reference's order */
enum { RT_ALGO_ONOFF = 0, RT_ALGO_FLAT = 1, RT_ALGO_PATHTRACING = 2, RT_ALGO_POINTLIGHT = 3 };

/* Arithmetic type of the traced path.  F32: fp32 throughout (path tracing's production arithmetic).
 * F64: fp64 without multiply-add fusion, the reference's own decisions (hit index bit-exact).
 * HYBRID (deterministic renderers, perspective camera, RT_ACCEL_NONE): an fp32 sweep that provably
 * never drops a sphere the reference hits, then the F64 code on the few spheres that pass — the F64
 * image bit for bit, at the speed of the fp32 sweep.
 * AUTO = F32 for path tracing; HYBRID for the deterministic renderers where it applies, else F64. */
enum { RT_PRECISION_AUTO = 0, RT_PRECISION_F32 = 1, RT_PRECISION_F64 = 2, RT_PRECISION_HYBRID = 3 };

/* Path-tracer kernel. MEGA = one thread per pixel-sample walking the recursion of
 * render.py:99-139 depth-first in the reference's own order; WARP = warp-cooperative
 * wavefront: 32 lanes drain a shared-memory stack of scatter records, children compacted
 * with ballots so that lanes stay full whatever the branching of single samples. */
enum { RT_VARIANT_AUTO = 0, RT_VARIANT_MEGA = 1, RT_VARIANT_WARP = 2 };

/* How the scatter/roulette random numbers are organised (path tracing only).
 * STREAMS: sample k owns PCG(init_state = pt_state, init_seq = (pt_inc >> 1) + k): the
 *          image does not depend on how samples are spread over threads or GPUs.
 * REPLAY : sample k starts from replay_states[k] with increment pt_inc and draws in the
 *          reference's order (MEGA variant only). Feeding the states the sequential
 *          reference stream has at the start of every sample reproduces the reference
 *          image itself, not just its distribution. */
enum { RT_RNG_STREAMS = 0, RT_RNG_REPLAY = 1 };

/* Multi-GPU partition of one image. SPP: rank r traces the strata s with
 * s % part_count == r of every pixel; ROWS: rank r traces the rows y with
 * y % part_count == r (interleaved: cost per row varies 1..85 rays/sample on demo.txt).
 * Every rank writes a full-size image holding its share (already scaled by 1/S^2; rows it
 * does not own are zero), so one sum over ranks is the final image. */
enum { RT_PART_NONE = 0, RT_PART_SPP = 1, RT_PART_ROWS = 2 };

/* Where RT_PART_ROWS stores the rows a rank owns.  FULL: in place in a full-size image (the other rows are
 * zero).  COMPACT: densely, [owned rows][width][3] — the slab an all-gather moves; rt_render() (host
 * buffers) then copies the slab's rows to rows rank, rank + count, ... of the caller's FULL-SIZE host image
 * and touches nothing else, so that ranks sharing one page-locked host image fill it together without any
 * device-side exchange. */
enum { RT_ROWS_FULL = 0, RT_ROWS_COMPACT = 1 };
#define RT_MAX_PEERS 8

/* Content of the optional int32[H][W] side image: the shape hit by the last sample of the pixel
 * (-1 = miss), or the number of rays (closest-hit + shadow queries) this rank traced for the
 * pixel — the divergence map of the scene. */
enum { RT_HIT_SHAPE = 0, RT_HIT_RAY_COUNT = 1 };

/* RT_ACCEL_NONE: the reference's algorithm, a loop over every shape per ray (world.py:55-64); this is
 * the path the FP32 roofline figures are quoted on.  RT_ACCEL_BVH: a bounding-volume hierarchy over
 * the spheres skips those whose box the ray misses — identical images (same per-shape tests, same
 * tie rule, conservative culling), O(log N) instead of O(N) work per ray; reported separately. */
enum { RT_ACCEL_NONE = 0, RT_ACCEL_BVH = 1 };

enum {
  RT_OK = 0,
  RT_ERR_INVALID = -1,   /* bad argument / unsupported combination */
  RT_ERR_CUDA = -2,      /* CUDA runtime error, text in rt_last_error() */
  RT_ERR_NO_DEVICE = -3, /* no CUDA device: there is no CPU fallback */
  RT_ERR_OVERFLOW = -4   /* device-side work stack overflow (reported, never silent) */
};

/* Pigment.get_color, materials.py:58 / :70-82 / :96-100 */
typedef struct rt_pigment {
  int32_t kind;
  int32_t num_of_steps;   /* checkered */
  int32_t tex_width;      /* image */
  int32_t tex_height;
  int64_t tex_offset;     /* first texel of this image inside rt_scene_desc.texels, in texels */
  double color1[3];       /* uniform: the colour; checkered: color1 */
  double color2[3];       /* checkered: color2 */
} rt_pigment;

/* Material, materials.py:199-204 */
typedef struct rt_material {
  int32_t brdf_kind;
  int32_t brdf_pigment;     /* index into pigments */
  int32_t emitted_pigment;  /* index into pigments */
  int32_t _pad;
  double threshold_angle_rad; /* SpecularBRDF.eval only, materials.py:158-173 */
} rt_material;

/* PointLight, lights.py:25-39 */
typedef struct rt_light {
  double position[3];
  double color[3];
  double linear_radius;
} rt_light;

/* World (world.py:36-49) flattened; shapes keep the order of World.shapes because
 * ray_intersection lets the FIRST shape win ties (world.py:62, strict '<'). */
typedef struct rt_scene_desc {
  int32_t n_shapes;
  int32_t n_materials;
  int32_t n_pigments;
  int32_t n_lights;
  const int32_t* shape_kind;      /* [n_shapes] */
  const int32_t* shape_material;  /* [n_shapes] index into materials */
  const double* shape_m;          /* [n_shapes][12] Transformation.m rows 0..2 */
  const double* shape_invm;       /* [n_shapes][12] Transformation.invm rows 0..2 */
  const rt_material* materials;
  const rt_pigment* pigments;
  const rt_light* lights;
  int64_t n_texels;
  const double* texels;           /* [n_texels][3] RGB, image rows top to bottom (HdrImage.pixels order) */
} rt_scene_desc;

/* Camera, camera.py:42-124 */
typedef struct rt_camera {
  int32_t kind;
  int32_t _pad;
  double screen_distance; /* perspective only */
  double aspect_ratio;
  double m[12];           /* camera Transformation.m rows 0..2 */
} rt_camera;

typedef struct rt_render_params {
  int32_t width;
  int32_t height;
  int32_t samples_per_side; /* 0 = one ray through the pixel centre, no RNG (imagetracer.py:103) */
  int32_t algorithm;
  rt_camera camera;
  double background[3];     /* Renderer.background_color */
  double onoff_color[3];    /* OnOffRenderer.color */
  double ambient[3];        /* PointLightRenderer.ambient_color */
  int32_t num_of_rays;      /* PathTracer */
  int32_t max_depth;
  int32_t rr_limit;         /* PathTracer.russian_roulette_limit */
  int32_t rng_mode;
  /* ImageTracer.pcg as it is when fire_all_rays starts: sample k (row-major pixels, then
   * strata rows, then strata columns) uses draws 2k and 2k+1 of this stream, u before v
   * (imagetracer.py:88-93). The device jumps ahead instead of drawing sequentially. */
  uint64_t aa_state;
  uint64_t aa_inc;
  /* PathTracer.pcg as it is when fire_all_rays starts (see RT_RNG_*). */
  uint64_t pt_state;
  uint64_t pt_inc;
  const uint64_t* replay_states; /* HOST pointer, [width*height*max(1,S)^2], RT_RNG_REPLAY only */
  int32_t part_mode;
  int32_t part_rank;
  int32_t part_count;
  int32_t variant;
  int32_t precision;
  int32_t out_f64;          /* 1: out_rgb is double[H][W][3] instead of float */
  int32_t hit_mode;         /* what out_hit_index receives: RT_HIT_SHAPE or RT_HIT_RAY_COUNT */
  int32_t accel;            /* RT_ACCEL_*: how World.ray_intersection / is_point_visible find their shapes */
  int32_t rows_layout;      /* RT_ROWS_* (RT_PART_ROWS only) */
  /* n_peer_images > 0 (rt_render_device, RT_PART_ROWS, RT_ROWS_FULL, fp32 image): the render kernel stores
   * every finished pixel into ALL of peer_images[0 .. n) — full-size images of the ranks of one node,
   * mapped into this process (CUDA IPC / symmetric memory; peer_images[part_rank] is this rank's own) —
   * instead of d_out_rgb: the exchange of the row split happens inside the kernel, pixel by pixel over
   * NVLink, and needs no collective afterwards (only a barrier before anyone reads). */
  int32_t n_peer_images;
  void* peer_images[RT_MAX_PEERS];
} rt_render_params;

typedef struct rt_stats {
  uint64_t rays_closest;  /* World.ray_intersection calls, world.py:51 */
  uint64_t rays_shadow;   /* World.is_point_visible calls, world.py:71 */
  uint64_t samples;       /* Renderer.__call__ invocations from fire_all_rays */
  float kernel_ms;        /* CUDA events around the render kernels, on the launch stream */
  float total_ms;         /* kernel_ms + device->host copy when the call does one */
  int32_t variant_used;
  int32_t precision_used;
  int32_t n_launches;     /* kernels of this library launched by the call */
  int32_t overflow;       /* non-zero: a warp work stack overflowed, image is invalid */
} rt_stats;

/* One closest hit, mirrors HitRecord (hitrecord.py:27-46) + the index World's loop would report */
typedef struct rt_hit {
  int32_t shape;          /* index in World.shapes, -1 = miss */
  int32_t material;
  double t;
  double world_point[3];
  double normal[3];       /* normalised, as World.ray_intersection returns it (world.py:66-67) */
  double uv[2];
} rt_hit;

typedef struct rt_scene rt_scene;

/* ---- device / errors ---- */
int rt_api_version(void);
int rt_device_count(void);
int rt_set_device(int device);
const char* rt_last_error(void);

/* ---- scene: replaces the object graph walked by World.ray_intersection ---- */
int rt_scene_create(const rt_scene_desc* desc, rt_scene** out);
void rt_scene_destroy(rt_scene* scene);

/* Animation: new Transformation.m / .invm (double[n][12] each, rows 0..2) for the shapes
 * [first, first + n) of World.shapes; everything else of the scene stays resident.  Replaces the
 * reference's per-frame re-parse with `--declare-float clock:VALUE` (main.py:122-128,
 * scene_file.py:654-675) for frames where only transformations change.  Enqueued on `stream`
 * (cudaStream_t as void*, NULL = default), after the renders already enqueued there. */
int rt_scene_update_transforms(rt_scene* scene, int32_t first, int32_t n, const double* m,
                               const double* invm, void* stream);

/* The sphere hierarchy of RT_ACCEL_BVH as rt_render builds it, computed on the HOST (needs no device; used
 * by the CPU test-suite to check the tree's invariants and the conservativeness of its padded boxes).
 * m: double[n_spheres][12], Transformation.m rows 0..2 of the spheres.  nodes_out: float[cap_nodes][16]
 * (per node: lo0.xyz hi0.xyz lo1.xyz hi1.xyz, then four int32 bit patterns ref0 ref1 0 0; a reference
 * >= 0 is an inner node, < 0 a leaf -(1 + first * 64 + (count - 1)) into prims_out[n_spheres]).
 * Returns RT_ERR_INVALID if cap_nodes is too small (n_spheres nodes always suffice). */
int rt_bvh_build_host(const double* m, int32_t n_spheres, float* nodes_out, int32_t cap_nodes,
                      int32_t* prims_out, int32_t* n_nodes, int32_t* depth);

/* ---- the hot path: ImageTracer.fire_all_rays(renderer) ---- */
/* Host buffers: out_rgb float[H][W][3] (or double if out_f64), out_hit_index int32[H][W]
 * (optional; shape hit by the LAST sample of each pixel, -1 = miss). Blocking. */
int rt_render(rt_scene* scene, const rt_render_params* params, void* out_rgb,
              int32_t* out_hit_index, rt_stats* stats);
/* The same image from ALL the devices of a node in one call, one process (SURVEY §8b/e; the reference has
 * no parallelism to replace — this is fire_all_rays again): scenes[i] = rt_scene_create() of the same World
 * with device i current (rt_set_device).  Device i traces the interleaved rows i, i + n, ... and copies them
 * into out_rgb / out_hit_index; the image is bit-identical to rt_render's on one device.  params->part_mode
 * must be RT_PART_NONE.  stats: counters summed over the devices, kernel_ms / total_ms = the slowest device.
 * Page-lock the host image (rt_host_register) so that the copies of the devices overlap. */
int rt_render_multi(rt_scene* const* scenes, int32_t n_scenes, const rt_render_params* params, void* out_rgb,
                    int32_t* out_hit_index, rt_stats* stats);
/* Same with DEVICE buffers on a caller stream (cudaStream_t passed as void*; NULL = default
 * stream). Returns after enqueueing; call rt_render_finish() to synchronise the stream and
 * collect the counters. */
int rt_render_device(rt_scene* scene, const rt_render_params* params, void* d_out_rgb,
                     int32_t* d_out_hit_index, void* stream);
int rt_render_finish(rt_scene* scene, void* stream, rt_stats* stats);

/* ---- path tracing with a per-pixel error map and noise-targeted passes ----
 * Pass p (p = 0, 1, ...) of a pixel is that pixel of the (p+1)-th consecutive fire_all_rays with the same
 * tracer and renderer: jitter stream advanced by p * 2 * W * H * S^2 draws, pt_state by p PCG steps, sample
 * indices k = pix * S^2 + s.  Pass 0 traces every pixel; every further pass traces, in ascending order, the
 * pixels whose relative error e = max_c SE_c / max(mean_c, error_floor) is still above target_error and that
 * have passes left.  A pass's squared standard error comes from batch sums of its S^2 samples (sample s in batch
 * s mod B' with B' = 32 / G, G = pixels per warp task, B = min(S^2, B') batches); `estimator` picks the formula:
 *   RT_ERR_EST_BATCH  (default): SE^2 = sum_b (T_b - n_b m)^2 / (n_b (B - 1) S^2), unbiased for independent
 *                     samples, too large where stratification removes variance (it treats strata as independent);
 *   RT_ERR_EST_PAIRED (S even): collapsed strata, SE^2 = sum_j (T_2j - T_2j+1)^2 / S^4 over j < B / 2.  Batches
 *                     2j and 2j + 1 hold horizontally adjacent strata in equal numbers, so each difference sums
 *                     pair differences; the estimate is conservative and tight where radiance is smooth across
 *                     two strata, with B / 2 degrees of freedom (half the batch estimator's).
 * A pixel with P passes reports mean = (sum of pass means,
 * fp32, in pass order) / P, SE = sqrt(sum of SE^2) / P and P * S^2 samples; with P = 1 the mean is rt_render's
 * pixel bit for bit.  Path tracing, WARP variant (AUTO picks it), fp32, S >= 2, RT_PART_NONE, RT_RNG_STREAMS,
 * no peer images, no out_f64, a known estimator (RT_ERR_EST_PAIRED: S even): anything else is RT_ERR_INVALID.
 * Host buffers, blocking; one device. */
enum { RT_ERR_EST_BATCH = 0, RT_ERR_EST_PAIRED = 1 };
typedef struct rt_adaptive_params {
  double target_error;        /* e threshold; <= 0: one pass, error map only */
  double error_floor;         /* absolute radiance floor of the relative error (> 0) */
  int32_t max_passes;         /* >= 1; pass p uses the PCG states defined above */
  int32_t estimator;          /* RT_ERR_EST_*: how a pass's SE^2 is formed (0 = batch) */
} rt_adaptive_params;
typedef struct rt_adaptive_stats {
  uint64_t rays_closest, rays_shadow, samples;
  float kernel_ms;            /* CUDA events around all passes (render, combine, select) and the final kernel */
  float total_ms;             /* the whole call, device->host copies included */
  int32_t passes;             /* passes actually run */
  int32_t n_launches;
  int64_t pixels_in_pass[16]; /* first 16 passes: list length traced in each */
  int32_t overflow;           /* non-zero: a warp work stack overflowed, the image is invalid (RT_ERR_OVERFLOW) */
  int32_t _pad;
} rt_adaptive_stats;
/* out_rgb float[H][W][3] mean; out_err float[H][W][3] SE (optional); out_samples int32[H][W] (optional) */
int rt_render_adaptive(rt_scene* scene, const rt_render_params* params, const rt_adaptive_params* ap,
                       float* out_rgb, float* out_err, int32_t* out_samples, rt_adaptive_stats* stats);
/* The same passes, scheduled by a sample budget B = sample_budget (total samples) instead of a threshold.  Passes,
 * PCG states, the pass values, the reported mean / SE / samples and estimator mean what they mean above; M =
 * ap->max_passes (>= 1); target_error >= 0 (finite) only says which pixels may be traced again.
 *   Pass 0 traces every pixel and needs B >= W*H*S^2.  Each pixel holds its e = max_c SE_c / max(mean_c,
 *   error_floor) (the fp32 value the threshold mode compares) from the last pass that traced it; the candidates
 *   are the pixels with e > target_error (target 0: every pixel with any error).  After pass p, if p + 1 < M, with
 *   Q = floor((B - samples spent) / S^2), C = the number of candidates and r = M - 1 - p, the next pass traces
 *       K = min(C, Q, max(ceil(C / 2), ceil(Q / r)))
 *   pixels: the first K in the order (e descending, pixel index ascending), listed in ascending pixel order.  The
 *   call stops when K = 0 or after M passes.  A pixel may skip passes; pass p of a pixel is always that pixel of
 *   the (p+1)-th fire_all_rays.
 * So every pass after the first traces at least half of the candidates the budget allows, the last allowed pass
 * spends what is left, no pixel gets more than M*S^2 samples, and stats->samples <= B with B - samples < S^2
 * unless the candidates ran out first.  The same scope as rt_render_adaptive, plus B >= W*H*S^2 and a finite
 * target_error >= 0; anything else is RT_ERR_INVALID. */
int rt_render_adaptive_budget(rt_scene* scene, const rt_render_params* params, const rt_adaptive_params* ap,
                              int64_t sample_budget, float* out_rgb, float* out_err, int32_t* out_samples,
                              rt_adaptive_stats* stats);
/* The same passes, scheduled by a ray budget R = ray_budget (>= 0): closest-hit rays, the quantity
 * stats->rays_closest counts.  Passes, PCG states, the pass values, the reported mean / SE / samples and estimator
 * mean what they mean above; M = ap->max_passes (>= 1); target_error >= 0 (finite) and error_floor as in the
 * sample-budget mode.
 *   Pass 0 traces every pixel, whatever R is.  Each pixel holds, from the last pass that traced it, its pass count P,
 *   its e (as above) and n = the closest-hit rays traced for it over all its passes.  Its predicted cost of one more
 *   pass is w = ceil(n / P) (>= S^2: every sample traces its primary ray).  A candidate (e > target_error) has the key
 *       fmaxf(__fdiv_rn(e, __fsqrt_rn(__fmul_rn((float)(P + 1), (float)w))), FLT_MIN)   (= e / sqrt((P + 1) w))
 *   which ranks by e^2 / ((P + 1) w), the drop in relative variance one more pass buys per predicted ray; FLT_MIN
 *   (a normal number: flush-to-zero cannot drop it) keeps every candidate's key above a non-candidate's 0.  After pass
 *   p, if p + 1 < M, with R_left = R - the closest-hit rays spent so far (read on the device; R_left <= 0: an empty
 *   pass), W_c = the sum of w over the candidates and r = M - 1 - p, the spend target is
 *       T = min(R_left, max(ceil(W_c / 2), ceil(R_left / r)))
 *   and the next pass traces the longest prefix of the order (key descending, pixel index ascending) whose sum of w
 *   is <= T, listed in ascending pixel order.  The call stops when that prefix is empty or after M passes.
 * So every pass after the first has a predicted cost within what is left of the budget, and while the budget lasts
 * covers at least half of the candidates' predicted cost less one pixel's; no pixel gets more than M*S^2 samples;
 * and the rays spent exceed R only by how far passes' actual rays exceeded their prediction, or because pass 0 alone
 * costs more than R.  out_rays int64[H][W] (optional): the closest-hit rays each pixel received (they sum to
 * stats->rays_closest).  The same scope as rt_render_adaptive, plus R >= 0 and a finite target_error >= 0; anything
 * else is RT_ERR_INVALID. */
int rt_render_adaptive_rays(rt_scene* scene, const rt_render_params* params, const rt_adaptive_params* ap,
                            int64_t ray_budget, float* out_rgb, float* out_err, int32_t* out_samples, int64_t* out_rays,
                            rt_adaptive_stats* stats);

/* ---- Renderer.__call__(ray) for explicit rays (render.py:52,65,99,157) ----
 * rays: double[n][8] = origin xyz, dir xyz, tmin, tmax; depth int32[n] (NULL = 0).
 * pcg_state_inc: {state, inc} of PathTracer.pcg, read and written back (rays are traced
 * one after the other on ONE stream in the reference's draw order). */
int rt_trace_rays(rt_scene* scene, const rt_render_params* params, const double* rays,
                  const int32_t* depth, int32_t n, uint64_t* pcg_state_inc, double* out_rgb);

/* ---- probes used by the known-answer tests (one per reference function) ---- */
/* World.ray_intersection, world.py:51-69 (normalize_normal = 1), or the raw record of the winning
 * Shape.ray_intersection, shapes.py:97-131 / :163-189 (normalize_normal = 0) */
int rt_intersect(rt_scene* scene, int32_t precision, int32_t normalize_normal, const double* rays,
                 int32_t n, rt_hit* out);
/* World.is_point_visible(point, observer_pos), world.py:71-80; pairs double[n][6] = point, observer */
int rt_is_point_visible(rt_scene* scene, int32_t precision, const double* pairs, int32_t n,
                        uint8_t* out);
/* ImageTracer.fire_ray for every sample of the image, in sample order; out double[n][8] */
int rt_camera_rays(const rt_render_params* params, int32_t precision, double* out_rays);
/* Camera.fire_ray(u, v), camera.py:59-78 / :103-124: uv double[n][2] -> rays double[n][8] */
int rt_camera_fire(const rt_camera* camera, int32_t precision, const double* uv, int32_t n,
                   double* out_rays);
/* PCG.random, pcg.py:43-58: n draws from {state, inc}; state_inc is updated */
int rt_pcg_draw(uint64_t* state_inc, int32_t n, uint32_t* out);
/* PCG.__init__, pcg.py:29-41 evaluated on the device */
int rt_pcg_seed(uint64_t init_state, uint64_t init_seq, uint64_t* state_inc);
/* Pigment.get_color: uv double[n][2] -> rgb double[n][3] */
int rt_pigment_color(rt_scene* scene, int32_t pigment, int32_t precision, const double* uv,
                     int32_t n, double* out_rgb);
/* BRDF.scatter_ray (materials.py:132-152, :175-196) for material `material`:
 * in double[n][9] = incoming dir, interaction point, normal; out rays double[n][8];
 * draws come sequentially from {state, inc}. */
int rt_scatter(rt_scene* scene, int32_t material, int32_t precision, const double* in,
               int32_t n, uint64_t* state_inc, double* out_rays);
/* create_onb_from_z, geometry.py:247-262: normals double[n][3] -> double[n][9] = e1,e2,e3 */
int rt_onb(int32_t precision, const double* normals, int32_t n, double* out);

/* ---- tone mapping: the step after the render (main.py:209-215, pfm2png main.py:226-230) ----
 * rgb: float[n_pixels][3] in HdrImage.pixels order; on_device != 0 means every buffer of the call is
 * a DEVICE pointer and the kernels run on `stream` (cudaStream_t as void*, NULL = default stream);
 * otherwise host buffers are copied in and out.  Both calls synchronise the stream before returning.
 * Arithmetic is fp64 in the reference's operation order on the fp32 pixel values (what the reference
 * computes on an image read back from a PFM file). */
typedef struct rt_tonemap_stats {
  double luminosity;  /* the average luminosity used (computed or passed in) */
  float lum_ms;       /* CUDA events around the luminosity kernel (0 if luminosity was passed in) */
  float map_ms;       /* CUDA events around the normalise/clamp/quantise kernel */
  float total_ms;     /* whole call on the stream, copies included */
  int32_t n_launches;
} rt_tonemap_stats;
/* HdrImage.average_luminosity(delta), hdrimages.py:120-128: 10 ** mean(log10(delta + luminosity)) */
int rt_average_luminosity(const float* rgb, int64_t n_pixels, double delta, int32_t on_device,
                          void* stream, double* out);
/* One pass over the image doing any of: HdrImage.normalize_image(factor, luminosity)
 * (hdrimages.py:130-140, flag RT_TONE_NORMALIZE), clamp_image() (hdrimages.py:142-147, flag
 * RT_TONE_CLAMP) -> out_hdr float[n][3] (optional), and write_ldr_image's int(255 * c ** (1 / gamma))
 * of the result (hdrimages.py:160-165) -> out_ldr uint8[n][3] (optional).  With RT_TONE_NORMALIZE,
 * luminosity == 0 (or NaN) is the reference's `if not luminosity`: the image's own
 * average_luminosity() is computed first.  main.py:209-215 = flags 3 with out_ldr. */
enum { RT_TONE_NORMALIZE = 1, RT_TONE_CLAMP = 2 };
int rt_tone_map(const float* rgb, int64_t n_pixels, int32_t flags, double factor, double luminosity, double gamma,
                int32_t on_device, void* stream, float* out_hdr, uint8_t* out_ldr,
                rt_tonemap_stats* stats);

/* ---- host buffers ----
 * Page-locks / unlocks a caller-owned host buffer (cudaHostRegister) so that rt_render's final
 * device->host copy of the image runs at full PCIe speed.  Optional: pageable buffers work too. */
int rt_host_register(void* ptr, uint64_t bytes);
int rt_host_unregister(void* ptr);

/* ---- measurement aid: FP32 FMA roofline denominator measured on this device ----
 * Runs a register-resident FFMA chain kernel (8 independent accumulators per thread, grid sized to
 * fill every SM) and reports achieved TFLOP/s (2 flops per FMA) and the kernel time. */
int rt_bench_ffma(int32_t iterations, double* tflops, float* ms);
/* Same with DFMA chains: the denominator for the fp64 share of the F64 / HYBRID kernels (which, compiled
 * without multiply-add fusion like the reference's arithmetic, can reach half of it in flops). */
int rt_bench_dfma(int32_t iterations, double* tflops, float* ms);

#ifdef __cplusplus
}
#endif
#endif
