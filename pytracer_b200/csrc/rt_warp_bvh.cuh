// rt_warp_bvh.cuh — PathTracer (render.py:99-139) over the sphere hierarchy (accel = RT_ACCEL_BVH).
//
// Same estimator, same scatter records, same random streams as k_pt_warp (rt_warp.cuh): a warp owns a
// task (a few pixels x their strata) and a LIFO stack of scatter records in shared memory.  What changes
// is the schedule.  Walking a tree takes a different number of steps for every ray — a ray that leaves
// towards the sky is done after three nodes, one that skims the sphere field visits a hundred — so a
// warp that traces 32 rays in lock step and waits for the slowest keeps 5 of its 32 lanes busy
// (measured, BASELINE config 4: smsp__thread_inst_executed_per_inst_executed = 5.1).  Here every lane
// keeps its own ray and its own walk (rt_bvh.cuh: BvhWalk) across iterations of the warp's loop:
//
//   refill   lanes without a ray take the next owed rays off the record stack (or the next primaries)
//   walk     lanes with a ray advance their walk — box steps of all descending lanes together, then the
//            sphere tests of all lanes that reached a leaf together (rt_bvh.cuh) — until the walks still
//            going number `refill_at` or fewer and there is something to refill the others with
//   shade    lanes whose walk has ended scan the planes, shade, accumulate and push their record
//
// i.e. persistent traversal with dynamic ray fetch at warp scope, with the record stack as the pool.
// Pixel sums are kept as acc[slot][channel][lane] columns in shared memory (lane-private adds: no
// conflicts, no atomics), reduced over lanes when the task ends.
#pragma once
#include "rt_warp.cuh"

// Where a warp's scatter records live.  Shared memory (round 1) costs 7.7 KB per warp and, with the walk
// stacks, holds the kernel to two blocks (16 warps) per SM — at 4 warps per scheduler the issue slots were
// 52 % busy with `long_scoreboard` and `wait` on top (profiles/r2_c4_bvh_scaled4_full.csv): a latency-bound
// kernel short of warps.  A record is read once per owed ray and written once per scattering hit, a few
// bytes per hundred instructions of walking, so the stacks can live in GLOBAL memory (L2-resident, ld.cg /
// st.cg) and the shared memory goes to a third block per SM.
#ifndef RT_BVH_REC_GLOBAL
#define RT_BVH_REC_GLOBAL 1
#endif
#ifndef RT_BVH_MINB
#define RT_BVH_MINB (RT_BVH_REC_GLOBAL ? 3 : 2)
#endif
RT_DEV float4 rec_ld(const float4* p) { return RT_BVH_REC_GLOBAL ? __ldcg(p) : *p; }
RT_DEV void rec_st(float4* p, float4 v) { if (RT_BVH_REC_GLOBAL) __stcg(p, v); else *p = v; }
RT_DEV ScatterRec rec_load(const ScatterRec* r) {
  ScatterRec v;
  const float4* p = reinterpret_cast<const float4*>(r);
  v.a = rec_ld(p); v.b = rec_ld(p + 1); v.c = rec_ld(p + 2);
  return v;
}
RT_DEV void rec_store(ScatterRec* r, const ScatterRec& v) {
  float4* p = reinterpret_cast<float4*>(r);
  rec_st(p, v.a); rec_st(p + 1, v.b); rec_st(p + 2, v.c);
}
struct WarpBvhCfg {
  ScatterRec* rec_pool;  // RT_BVH_REC_GLOBAL: (cap + 1) records per resident warp
  WarpCfg w;
  int refill_at;      // leave the walk phase when at most this many walks are still going
  int inner_min;      // leave the box-test loop for the sphere-test loop when at most this many lanes are descending
  int stack_entries;  // per-lane walk stack in shared memory (tree depth + 1)
  int tree_bytes;     // > 0: nodes + leaf index list are copied to shared memory (w.shape_bytes holds the size)
  int n_nodes, n_prims;
};

// ERR: error-map instantiation, as k_pt_warp's (rt_warp.cuh err_batch_add)
template <bool ERR = false>
__global__ void __launch_bounds__(RT_WARP_MAX_THREADS, RT_BVH_MINB)
k_pt_warp_bvh(const __grid_constant__ SceneView<float> sc, const __grid_constant__ RenderArgs a,
              const __grid_constant__ WarpBvhCfg bcfg, const __grid_constant__ ErrArgs ea) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const WarpCfg& cfg = bcfg.w;
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  BvhSrc tree = bvh_global_src(sc);
  if (bcfg.tree_bytes > 0) {  // a small tree lives in shared memory: node fetches at 30 cycles instead of an L2 round trip
    stage_bytes(smem_raw, sc.bvh_nodes, (size_t)bcfg.n_nodes * 64);
    stage_words(smem_raw + (size_t)bcfg.n_nodes * 64, sc.bvh_prims, bcfg.n_prims * 4);
    __syncthreads();
    tree.nodes = reinterpret_cast<const float4*>(smem_raw);
    tree.prims = reinterpret_cast<const int32_t*>(smem_raw + (size_t)bcfg.n_nodes * 64);
  }
  unsigned char* wbase = smem_raw + cfg.shape_bytes + warp * cfg.per_warp_bytes;
  ScatterRec* stack = RT_BVH_REC_GLOBAL ? bcfg.rec_pool + ((size_t)blockIdx.x * (blockDim.x >> 5) + warp) * (size_t)(cfg.cap + 1)
                                        : reinterpret_cast<ScatterRec*>(wbase);
  ScatterRec* cur = stack + cfg.cap;
  int* slot_rays = RT_BVH_REC_GLOBAL ? reinterpret_cast<int*>(wbase) : reinterpret_cast<int*>(cur + 1);  // [32]
  float* acc = reinterpret_cast<float*>(slot_rays + 32);  // [G][3][32]
  float2* walk_stacks = reinterpret_cast<float2*>(acc + cfg.group * 96);  // [stack_entries][32]
  float* bsum = reinterpret_cast<float*>(walk_stacks + bcfg.stack_entries * 32);  // ERR: [32][3] batch sums
  // (ERR: each pixel's count goes to ea.err_rays instead of the side image)
  const bool count_rays = ERR ? ea.err_rays != nullptr : a.out_hit != nullptr && a.hit_mode == RT_HIT_RAY_COUNT;
  const float* planes = sc.invm + 12 * (size_t)sc.n_spheres;
  const int n_planes = sc.n_shapes - sc.n_spheres;

  const PixelMap pm = ERR ? make_pixel_map_list(a, ea) : make_pixel_map(a);
  auto locate = [&](long long p, int& col, int& row) { if (ERR) locate_listed(pm, ea, p, col, row); else pm.locate(p, col, row); };
  const int N = a.num_of_rays;
  const int S2 = a.S > 0 ? a.S * a.S : 1;
  const int G = cfg.group, L = cfg.per_pixel;
  auto div_n = [&](int x) -> int { return cfg.n_magic ? (int)(((unsigned)x * cfg.n_magic) >> 16) : (x >= N ? 1 : 0); };
  const float inv_n = cfg.inv_n, inv_spp = cfg.inv_spp;
  unsigned int n_rays = 0;  // warp-uniform
  bool overflow = false;

  while (true) {
    long long task = 0;
    if (lane == 0) task = (long long)atomicAdd(a.counters + CNT_TASK, 1ull);
    task = __shfl_sync(FULL, task, 0);
    if (task >= cfg.n_tasks) break;
    const long long p0 = task * G;
    const int task_prims = (int)min((long long)G, pm.n_pixels - p0) * L;
    for (int i = 0; i < 3 * G; ++i) acc[i * 32 + lane] = 0.f;
    slot_rays[lane] = 0;
    if (ERR) { for (int i = lane; i < 96; i += 32) bsum[i] = 0.f; }
    __syncwarp();

    // ---- per-lane state that lives across iterations
    bool busy = false, walking = false;
    Ray<float> ray;
    V3<float> thr = mk3<float>(1.f, 1.f, 1.f);
    uint64_t rng_state = 0;
    int slot = 0, depth = 0, origin = -1;
    int rslot = 0;  // ERR: the slot field of this ray's records, the batch (`slot` stays the pixel in the task)
    long long pix = -1;  // >= 0: a primary ray whose hit goes to out_hit[pix]
    float best_t = Num<float>::inf();
    int best = -1;
    BvhWalk<BvhSharedStack> walk;
    walk.stack.base = walk_stacks + lane;
    // ---- warp-uniform state
    int top = 0, cur_rem = 0, cur_done = 0, prim_next = 0;

    while (true) {
      // ---------------- refill: free lanes take rays, in lane order
      const unsigned free_mask = __ballot_sync(FULL, !busy);
      const int n_free = __popc(free_mask);
      const int rank = __popc(free_mask & lt_mask);
      if (prim_next < task_prims) {
        const int take = min(n_free, task_prims - prim_next);
        if (!busy && rank < take) {
          const int j = prim_next + rank;
          slot = j / L;
          const int ls = j - slot * L;
          if (ERR) rslot = slot * ea.err_bpp + err_batch_of(ea, ls);
          int col, row;
          locate(p0 + slot, col, row);
          const long long px = (long long)row * a.width + col;
          const int s = own_stratum(a, ls);
          const unsigned long long k = (unsigned long long)px * S2 + s;
          Pcg aa;
          aa.inc = a.aa_inc;
          aa.state = (a.S > 0) ? pcg_jump(a.aa_state, 2ull * k, a.jump) : 0;
          ray = primary_ray_mul(a, cfg.inv_w, cfg.inv_h, cfg.inv_s, col, row, s, aa);
          rng_state = pcg_seed(a.pt_state, (a.pt_inc >> 1) + k).state;
          thr = mk3<float>(1.f, 1.f, 1.f);
          depth = 0;
          origin = -1;
          pix = (ls == L - 1) ? pm.at(p0 + slot, col, row) : -1;
          busy = true;
        }
        prim_next += take;
        n_rays += (unsigned)take;
      } else {
        const long long avail = (long long)cur_rem + (long long)top * N;
        const int take = (int)min(avail, (long long)n_free);
        const bool get = !busy && rank < take;
        const int from_cur = min(cur_rem, take);
        ScatterRec rec;
        int child = 0;
        if (get) {
          if (rank < from_cur) {
            rec = rec_load(cur);
            child = cur_done + rank;
          } else {
            const int jj = rank - from_cur;
            const int r = div_n(jj);
            child = jj - r * N;
            rec = rec_load(&stack[top - 1 - r]);
          }
        }
        const int rest = take - from_cur;
        const int full = div_n(rest), part = rest - full * N;
        cur_rem -= from_cur;
        cur_done += from_cur;
        __syncwarp();  // every lane has read its record
        int new_top = top - full;
        if (part > 0) {  // the next record is only partly consumed: it becomes `cur`
          if (lane < 3) rec_st(reinterpret_cast<float4*>(cur) + lane, rec_ld(reinterpret_cast<const float4*>(&stack[new_top - 1]) + lane));
          new_top -= 1;
          cur_rem = N - part;
          cur_done = part;
        }
        __syncwarp();
        top = new_top;
        n_rays += (unsigned)take;
        if (get) {
          const int meta = __float_as_int(rec.a.w);
          slot = meta & 31;
          if (ERR) { rslot = slot; slot = (int)(((unsigned)rslot * ea.err_magic) >> 16); }  // the batch's pixel in the task
          depth = (meta >> 6) & 1023;
          origin = (int)((unsigned)meta >> 16);
          if (origin == 0xFFFF) origin = -1;
          thr = mk3<float>(rec.b.w, rec.c.x, rec.c.y);
          const uint64_t base = ((uint64_t)__float_as_uint(rec.c.w) << 32) | (uint64_t)__float_as_uint(rec.c.z);
          Pcg rng;
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
          rng_state = rng.state;
          pix = -1;
          busy = true;
        }
      }
      if (busy && !walking) {  // a ray taken just now: start its walk
        best_t = Num<float>::inf();
        best = -1;
        bvh_begin<float>(sc, ray, best_t, walk);
        walking = walk.ref != RT_BVH_DONE;
        if (count_rays) atomicAdd(&slot_rays[slot], 1);
      }
      if (__ballot_sync(FULL, busy) == 0u) break;  // nothing in flight and nothing left to take: the task is done

      // ---------------- walk
      const bool more_work = prim_next < task_prims || (long long)cur_rem + (long long)top * N > 0;
      while (true) {
        // box steps together: until the lanes still descending are few (the others wait at a leaf or are done)
        while (true) {
          const bool inner = walking && walk.ref >= 0;
          const unsigned mi = __ballot_sync(FULL, inner);
          if (__popc(mi) <= bcfg.inner_min && (mi == 0u || __ballot_sync(FULL, walking && walk.ref < 0) != 0u)) break;
          if (inner) bvh_inner_step(tree, walk);
        }
        // sphere tests together: one sphere per lane and round, until no lane is at a leaf
        while (true) {
          const bool leaf = walking && walk.ref < 0 && walk.ref != RT_BVH_DONE;
          if (__ballot_sync(FULL, leaf) == 0u) break;
          if (leaf) bvh_leaf_step<float>(sc, tree, ray, best_t, best, origin, walk);
        }
        walking = walking && walk.ref != RT_BVH_DONE;
        const unsigned m = __ballot_sync(FULL, walking);
        if (m == 0u) break;
        if (more_work && __popc(m) <= bcfg.refill_at) break;
      }

      // ---------------- shade the lanes whose walk has ended
      V3<float> contrib = mk3<float>(0.f, 0.f, 0.f);
      bool push = false;
      ScatterRec out;
      const bool done = busy && !walking;
      if (done) {
        scan_plane_block(planes, sc.n_spheres, n_planes, sc.orig, ray, best_t, best, origin);
        const bool found = best >= 0;
        if (pix >= 0 && a.out_hit && !count_rays) a.out_hit[pix] = found ? sc.orig[best] : -1;
        if (!found) {
          contrib = mk3<float>(thr.x * cfg.bg[0], thr.y * cfg.bg[1], thr.z * cfg.bg[2]);
        } else {  // lazy hit record, see k_pt_warp
          const DevMaterial& mat = sc.materials[sc.material[best]];
          const int mf = mat.flags;
          const bool sphere = best < sc.n_spheres;
          const Rows3 im = rows_at(sc.invm + 12 * (size_t)best);  // the arithmetic of k_pt_warp, operation for operation
          float u = 0.f, v = 0.f;
          if (depth >= a.max_depth) {
            if (!(mf & MAT_EMIT_BLACK)) {
              if (mf & MAT_UV_EMIT) local_uv<float>(local_hit_rows(im, ray, best_t), sphere, u, v);
              contrib = mul3(thr, pigment_color<float>(sc.pigments, mat.emitted_pigment, u, v));
            }
          } else {
            const bool scatters = !(mf & MAT_NO_SCATTER);
            LocalHit<float> lh;
            if (scatters || (mf & MAT_USES_UV)) lh = local_hit_rows(im, ray, best_t);
            if (mf & MAT_USES_UV) local_uv<float>(lh, sphere, u, v);
            if (!(mf & MAT_EMIT_BLACK)) contrib = mul3(thr, pigment_color<float>(sc.pigments, mat.emitted_pigment, u, v));
            if (scatters) {
              V3<float> hit_color = pigment_color<float>(sc.pigments, mat.brdf_pigment, u, v);
              const float lum = max3(hit_color);
              bool go_on = true;
              Pcg rng;
              rng.state = rng_state;
              rng.inc = a.pt_inc;
              if (depth >= a.rr_limit) {  // render.py:116-123
                const float q = fmaxf(0.05f, 1.f - lum);
                if (pcg_random_float<float>(rng) > q) hit_color = fast_rcp(1.f - q) * hit_color;
                else go_on = false;
              }
              if (go_on && lum > 0.f) {
                push = true;
                V3<float> point, normal;
                world_frame_rows(im, rows_at(sc.m + 12 * (size_t)best), lh, sphere, point, normal);
                const V3<float> nd = (mat.brdf_kind == RT_BRDF_DIFFUSE) ? normal : specular_dir<float>(ray.d, normal);
                const V3<float> w = inv_n * mul3(thr, hit_color);
                out.a = make_float4(point.x, point.y, point.z,
                                    __int_as_float((ERR ? rslot : slot) | (mat.brdf_kind << 5) | ((depth + 1) << 6) |
                                                   ((best < 0xFFFF ? best : 0xFFFF) << 16)));
                out.b = make_float4(nd.x, nd.y, nd.z, w.x);
                out.c = make_float4(w.y, w.z, __uint_as_float((uint32_t)rng.state), __uint_as_float((uint32_t)(rng.state >> 32)));
              }
            }
          }
        }
        float* colm = acc + (3 * slot) * 32 + lane;  // this lane's own column of the pixel's accumulator
        colm[0] += contrib.x; colm[32] += contrib.y; colm[64] += contrib.z;
        busy = false;
      }
      if (ERR) err_batch_add(bsum, rslot, done, contrib, lane);
      // ---------------- push the new records: one ballot gives every lane its slot
      const unsigned pmask = __ballot_sync(FULL, push);
      const int npush = __popc(pmask);
      if (top + npush > cfg.cap) {
        overflow = true;
      } else if (push) {
        rec_store(&stack[top + __popc(pmask & lt_mask)], out);
      }
      if (top + npush <= cfg.cap) top += npush;
      __syncwarp();
    }

    // ---------------- write the pixels of this task
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
        if (p < pm.n_pixels) {
          err_store(ea, L, bsum, g, p, mk3<float>(r * inv_spp, gr * inv_spp, b * inv_spp), lane);
          if (count_rays && lane == 0) ea.err_rays[p] = slot_rays[g];
        }
      } else if (lane == 0 && p < pm.n_pixels) {
        int col, row;
        pm.locate(p, col, row);
        store_pixel<float>(a, pm.at(p, col, row), mk3<float>(r * inv_spp, gr * inv_spp, b * inv_spp));
        if (count_rays) a.out_hit[pm.at(p, col, row)] = slot_rays[g];
      }
    }
    __syncwarp();
  }
  if (overflow) atomicExch(a.counters + CNT_OVERFLOW, 1ull);
  if (lane == 0 && n_rays) atomicAdd(a.counters + CNT_CLOSEST, (unsigned long long)n_rays);
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(a.counters + CNT_SAMPLES, cfg.n_samples);
}

template <bool ERR = false>
inline cudaError_t launch_pt_warp_bvh(const SceneView<float>& sc, const RenderArgs& a, cudaStream_t st,
                                      int sm_count, LaunchInfo* info, const char** why_not, int n_nodes, int n_prims, int tree_depth,
                                      ErrArgs ea = ErrArgs()) {
  PixelMap pm = ERR ? make_pixel_map_list(a, ea) : make_pixel_map(a);
  const int S2 = a.S > 0 ? a.S * a.S : 1;
  int L = S2;
  if (a.part_mode == RT_PART_SPP && a.part_count > 1)
    L = a.part_rank < S2 ? (S2 - a.part_rank + a.part_count - 1) / a.part_count : 0;
  if (pm.n_pixels == 0 || L == 0) return cudaSuccess;
  if (a.num_of_rays < 1) { *why_not = "num_of_rays must be >= 1"; return cudaErrorInvalidValue; }
  if (a.max_depth < 0 || a.max_depth >= 1023) { *why_not = "max_depth outside [0, 1022] is left to the mega variant"; return cudaErrorInvalidValue; }
  WarpBvhCfg b;
  WarpCfg& cfg = b.w;
  memset(&b, 0, sizeof(b));
  cfg.per_pixel = L;
  // tasks of about 32 samples over at most RT_ACC_LANES_MAX_GROUP pixels: enough owed rays on the stack to
  // refill lanes from, accumulator columns for every pixel of the task
  int group = (32 + L - 1) / L;
  if (group > RT_ACC_LANES_MAX_GROUP) group = RT_ACC_LANES_MAX_GROUP;
  if (group < 1) group = 1;
  cfg.group = group;
  cfg.rounds = (group * L + 31) / 32;
  cfg.n_tasks = (pm.n_pixels + group - 1) / group;
  // records alive: one per primary of the task, plus what 32 rays in flight can push per tree level (twice
  // that, since walks of different levels overlap); overflow is detected and reported, never silent
  const long long prims = (long long)group * L;
  long long cap = a.num_of_rays == 1 ? prims + 64 : prims + 32ll * (long long)a.max_depth + 32;
  if (cap < 96) cap = 96;
  b.stack_entries = tree_depth + 2;
  b.n_nodes = n_nodes;
  b.n_prims = n_prims;
  // the tree itself goes to shared memory while RT_BVH_MINB blocks still fit an SM with it
  const size_t tree_bytes = ((size_t)n_nodes * 64 + (size_t)n_prims * 4 + 15) / 16 * 16;
  const size_t limit = 200 * 1024;
  int warps = RT_WARP_MAX_THREADS / 32;
  size_t per_warp = 0, smem = 0;
  for (;; warps >>= 1) {
    per_warp = (RT_BVH_REC_GLOBAL ? 0 : (size_t)(cap + 1) * sizeof(ScatterRec)) + 32 * sizeof(int) + (size_t)group * 96 * sizeof(float) +
               (size_t)b.stack_entries * 32 * sizeof(float2) + (ERR ? 96 * sizeof(float) : 0);
    b.tree_bytes = ((tree_bytes + per_warp * warps + 1024) * RT_BVH_MINB <= 227 * 1024) ? (int)tree_bytes : 0;
    smem = b.tree_bytes + per_warp * warps;
    if (smem <= limit || warps == 1) break;
  }
  if (smem > limit) { *why_not = "max_depth needs a deeper work stack than shared memory holds"; return cudaErrorInvalidValue; }
  cfg.cap = (int)cap;
  cfg.per_warp_bytes = (int)per_warp;
  cfg.shape_bytes = b.tree_bytes;
  for (int k = 0; k < 3; ++k) cfg.bg[k] = (float)a.background[k];
  cfg.inv_n = 1.0f / (float)a.num_of_rays;
  cfg.inv_spp = 1.0f / (float)S2;
  cfg.n_magic = a.num_of_rays <= 1024 ? (65536u + (unsigned)a.num_of_rays - 1u) / (unsigned)a.num_of_rays : 0u;
  cfg.n_samples = (unsigned long long)pm.n_pixels * (unsigned long long)L;
  cfg.inv_w = 1.0 / (double)a.width;
  cfg.inv_h = 1.0 / (double)a.height;
  cfg.inv_s = a.S > 0 ? 1.0 / (double)a.S : 1.0;
  ea.err_bpp = 32 / cfg.group;
  ea.err_magic = (65536u + (unsigned)ea.err_bpp - 1u) / (unsigned)ea.err_bpp;
  if (ERR && (a.S < 2 || L != S2)) { *why_not = "the error map needs samples_per_side >= 2 and no partition"; return cudaErrorInvalidValue; }
  b.refill_at = 12;  // measured with 24 warps per SM (profiles/r2_bvh_sweep2.log): 8 | 12 | 16 | 20 | 24 -> 6.14 | 6.17 | 6.12 | 5.98 | 5.87 Grays/s
#ifdef RT_TUNING
  if (const char* env = getenv("RT_BVH_REFILL_AT")) b.refill_at = atoi(env);
#endif
  if (b.refill_at < 0) b.refill_at = 0;
  if (b.refill_at > 31) b.refill_at = 31;
  b.inner_min = 8;
#ifdef RT_TUNING
  if (const char* env = getenv("RT_BVH_INNER_MIN")) b.inner_min = atoi(env);
#endif
  if (b.inner_min < 0) b.inner_min = 0;
  if (b.inner_min > 31) b.inner_min = 31;

  cudaError_t e = cudaFuncSetAttribute(k_pt_warp_bvh<ERR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit);
  if (e != cudaSuccess) return e;
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pt_warp_bvh<ERR>, warps * 32, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  long long blocks = (long long)per_sm * sm_count;  // persistent: every block stays resident
  long long needed = (cfg.n_tasks + warps - 1) / warps;
  if (blocks > needed) blocks = needed;
  if (RT_BVH_REC_GLOBAL) {  // record stacks of all resident warps: one allocation per device, grown on demand
    static ScatterRec* pool[64] = {nullptr};
    static size_t pool_bytes[64] = {0};
    int dev = 0;
    e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const size_t bytes = (size_t)blocks * warps * (size_t)(cap + 1) * sizeof(ScatterRec);
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (bytes > pool_bytes[dev]) {
      if (pool[dev]) { e = cudaDeviceSynchronize(); if (e == cudaSuccess) e = cudaFree(pool[dev]); if (e != cudaSuccess) return e; }  // (rare: a larger frame than ever before)
      pool[dev] = nullptr; pool_bytes[dev] = 0;
      e = cudaMalloc((void**)&pool[dev], bytes);
      if (e != cudaSuccess) return e;
      pool_bytes[dev] = bytes;
    }
    b.rec_pool = pool[dev];
  }
  k_pt_warp_bvh<ERR><<<(unsigned)blocks, warps * 32, smem, st>>>(sc, a, b, ea);
  if (info) { info->n_launches += 1; info->variant = RT_VARIANT_WARP; }
  return cudaGetLastError();
}
