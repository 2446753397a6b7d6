// rt_kernels.cuh — the wavefront kernels (sm_100a) and their launch-time data layout.
//
// Data layout in HBM (one "pass" = a batch of 16x16 film tiles; DESIGN.md §3):
//   per path (never moves; a path's id encodes pixel and sample):
//     o_time[g]  float4  origin.xyz, time            (ray.rs:8-9)
//     d_t[g]     float4  dir.xyz, closest-hit t      (ray.rs:10, hitable.rs:52-55)
//     rad[g]     float4  radiance.xyz, -             (ray.rs:11)
//     thr[g]     float4  throughput.xyz, -           (ray.rs:12)
//     nrm0[g]    float4  depth-0 world normal.xyz, bits(slot0+1) (integrator.rs:161-169)
//     term[g]    u32     kind<<30 | depth<<20 | slot at termination (integrator.rs:178-203)
//   per tile, index queues (the "ray queue": what is compacted and partitioned is a 4-byte id):
//     q_live[ts*R + i]    live path ids in packet order           (film.rs:608-625)
//     q_key[ts*R + id]    object hit by path id at this depth, -1 = nothing (hitable.rs:203-209); indexed by PATH so that
//                         the kernel that produces a ray (raygen, shade_post) can already run the analytic spheres
//                         that precede the first SDF in the fold order
//     q_shade[ts*QS + s]  shading slots: per-object bins, each padded to x4 with -1
//                         (hitable.rs:94-133)
//   g = ts*R + id, id = (xl*th + yl)*spp + sample  — the reference's raygen order
//   `for x { for y { for samp { 4 lanes } } }` (film.rs:456-464).
//
// Kernel sequence of a pass: k_raygen, then per depth
//   k_scan_live -> k_extend_spheres / k_extend_march<V> (fold order of hitable.rs:177-198) -> k_bin_count, k_bin_scatter
//   -> k_normals<V> (one per SDF hitable) -> k_shade_pre -> k_shadow<V> (one per SDF hitable)
//   -> k_shade_post -> k_compact_count, k_compact_scatter;  finally k_resolve.
// The two march kernels and k_normals evaluate the distance field on TWO points per thread with the packed
// f32x2 arithmetic of sm_100a (rt_sdf2.cuh).
#pragma once
#include "rt_device.cuh"
#include "rt_sdf2.cuh"

namespace rt {

struct DevFrame {
  int W, H, tile_w, tile_h, samples, spp, max_bounces, vm;
  int ntx, nty, sets_1d, sets_2d;
  float t0, t1;
  const float* __restrict__ s1;   // [spp*sets_1d]
  const float* __restrict__ s2;   // [2*spp*sets_2d]
  const float* __restrict__ scramble;  // [W*H]
  const float* __restrict__ fis;  // [512]
};

struct PassBufs {
  int n_tiles;  // tiles in this pass
  int R;        // path slots per tile = tile_w*tile_h*spp
  int QS;       // shading-queue stride per tile = R + 4*n_hit
  const int* __restrict__ tile_ids;  // [n_tiles] global tile index
  float4* o_time;
  float4* d_t;
  float4* rad;
  float4* thr;
  float4* nrm0;
  uint32_t* term;
  int* q_live;
  int* q_key;
  int* q_shade;
  int* n_live;     // [n_tiles]
  int* n_slots;    // [n_tiles]
  int* bin_start;  // [n_tiles*(Scn::kMaxHit+1)]: bin starts of every hitable, row stride by scene type (rt_device.cuh)
  unsigned long long* counters;  // [8] stats
  // shading split (normals -> pre -> persistent shadow march -> post)
  float4* nrm;        // [paths] shading normal.xyz, offset_by of the current depth (hitable.rs:21-28)
  uint32_t* vis;      // [paths] bit i = light sample i of this depth is visible
  // shadow segments of the current depth, one queue per SDF hitable (ordinal j): entries [j*seg_cap, j*seg_cap + seg_count[j])
  float4* seg_a;      // start.xyz, max_dist
  float4* seg_b;      // dir.xyz, bits(path index g << 4 | light-sample bit)
  int* seg_count;     // [RAYN_MAX_SDF_HITABLES] segments pushed this depth, per SDF ordinal
  long long seg_cap;  // capacity of ONE queue
  float4* lc_c;       // [paths * lc_ns] unoccluded light contribution c.xyz and its denominator (pdf), per light sample of this depth
  float* lc_t;        // [paths * 8] volume rounds only: transmission to the scatter point (integrator.rs:122-126)
  int lc_ns;          // light samples per path per depth: 4, or 4 * (1 + vm) with volumetrics
  int* seg_cnt;       // [n_tiles * nseg * Scn::kMaxHit] scratch of the segmented queue kernels (k_bin_*, k_compact_*)
  // work lists of the slot-parallel kernels (k_scan_slots): row 0 = 128-slot blocks of every tile's shading queue, row 1 + j =
  // 128-slot blocks of the bin of SDF ordinal j; each row is an exclusive prefix over the tiles with the total at [n_tiles]
  int* slot_prefix;   // [(1 + RAYN_MAX_SDF_HITABLES) * prefix_stride]
  int prefix_stride;  // >= n_tiles + 1
};

enum { CNT_EXTEND_RAYS = 0, CNT_SHADE_LANES = 1, CNT_SHADOW_RAYS = 2, CNT_EVALS_EXTEND = 3, CNT_EVALS_SHADOW = 4,
       CNT_BULB_ITERS_EXTEND = 5, CNT_BULB_ITERS_SHADOW = 6, CNT_EVALS_NORMALS = 7, CNT_TRIPS_EXTEND = 8, CNT_TRIPS_SHADOW = 9, CNT_TOTAL = 10 };  // Mandelbulb iterations actually run (the count is data dependent)

// global work counters of the persistent kernels (RaynContext::d_work_ctr), zeroed by k_scan_live every depth
// (a run of spheres is numbered by the SDF hitables before it: runs are separated by SDFs, so there are at most 1 + n_sdf)
enum { WC_EXTEND = 0, WC_SHADOW = 1 /* + SDF ordinal */, WC_SEG_COUNT = 1 + RAYN_MAX_SDF_HITABLES /* + SDF ordinal */,
       WC_PRE = 1 + 2 * RAYN_MAX_SDF_HITABLES, WC_POST = WC_PRE + 1, WC_NORMALS = WC_POST + 1 /* + SDF ordinal */,
       WC_SPHERES = WC_NORMALS + RAYN_MAX_SDF_HITABLES /* + SDFs before the run */, WC_TOTAL = WC_SPHERES + RAYN_MAX_SDF_HITABLES + 1 };

#define TERM_NONE 0u
#define TERM_COLOR 1u
#define TERM_BACKGROUND 2u
// term word: kind (2 bits) | depth (8 bits) | shading slot (22 bits).  The low 30 bits are the film-accumulation key.
#define TERM_DEPTH_SHIFT 22
#define TERM_MAX_SLOTS (1 << TERM_DEPTH_SHIFT)
#define TERM_MAX_DEPTH 255

struct TileGeom {
  int x0, y0, tw, th, npaths;
};
RT_D TileGeom tile_geom(const DevFrame& fr, int tile_id) {
  TileGeom g;
  int tx = tile_id / fr.nty, ty = tile_id % fr.nty;  // film.rs:403-405: x-major
  g.x0 = tx * fr.tile_w;
  g.y0 = ty * fr.tile_h;
  int x1 = min(g.x0 + fr.tile_w, fr.W), y1 = min(g.y0 + fr.tile_h, fr.H);  // film.rs:406-409
  g.tw = x1 - g.x0;
  g.th = y1 - g.y0;
  g.npaths = g.tw * g.th * fr.spp;
  return g;
}

// Samples::sample_1d / sample_2d, sampler.rs:62-64,92-94
RT_D float samp1(const DevFrame& fr, int sample, float scramble, int set) {
  return dm::fract(__ldg(fr.s1 + sample + (size_t)fr.spp * set) + scramble);
}
RT_D float samp2(const DevFrame& fr, int dim, int sample, float scramble, int set) {
  return dm::fract(__ldg(fr.s2 + dim + (size_t)sample * 2 + (size_t)fr.spp * 2 * set) + scramble);
}

// same for a partially active warp (callers that returned early)
RT_D void warp_add_partial(unsigned long long* ctr, int v) {
  const unsigned m = __activemask();
  const int s = __reduce_add_sync(m, v);
  if ((int)(threadIdx.x & 31) == __ffs(m) - 1 && s) atomicAdd(ctr, (unsigned long long)s);
}
RT_D void warp_add(unsigned long long* ctr, int v) {  // full warp; one REDUX instead of a five-step shuffle tree
  v = __reduce_add_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(ctr, (unsigned long long)v);
}

// The head of the closest-hit fold (hitable.rs:177-198): t_max = 2 * WORLD_RADIUS (film.rs:556), then the first n_fold analytic
// spheres of the scene's compact sphere list (DevScene::sph, insertion order) - the spheres that precede the first SDF
// hitable, or ALL spheres for scenes whose single SDF is marched last (api.cu: fold_all; proof at k_extend_march).  Run by
// the kernel that PRODUCES the ray (origin and direction are in registers there), which removes one gather of every live
// ray per depth.  Static spheres only: a moving sphere is evaluated at the time of lane 0 of the extend packet, which is
// not known before compaction (k_extend_spheres handles that case).
template <class Scn>
RT_D void fold_head(const Scn& sc, int n_fold, f3 o, f3 d, float* closest, int* id) {
  float c = sc.rc.world_radius * 2.0f;
  int best = -1;
  for (int k = 0; k < n_fold; ++k) {
    const float t = sphere_hit_static(sc.sph[k], o, d, c);
    if (t < c) {
      c = t;
      best = sc.sph_idx[k];
    }
  }
  *closest = c;
  *id = best;
}

// ------------------------------------------------------------------------------------------
// K1 raygen: film.rs:456-529 + sample_uv :695-709 + camera.rs get_rays
// ------------------------------------------------------------------------------------------
template <class Scn>
__global__ void __launch_bounds__(256) k_raygen(const __grid_constant__ Scn sc, const DevFrame fr, const PassBufs pb, const int pre_n) {
  const int ts = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const TileGeom tg = tile_geom(fr, pb.tile_ids[ts]);
  if (i == 0) pb.n_live[ts] = tg.npaths;
  if (i >= tg.npaths) return;
  const int pl = i / fr.spp, s = i - pl * fr.spp;
  const int xl = pl / tg.th, yl = pl - xl * tg.th;
  const int x = tg.x0 + xl, y = tg.y0 + yl;
  const float scramble = __ldg(fr.scramble + x + (size_t)y * fr.W);
  const float fx = fis_sample(fr.fis, samp2(fr, 0, s, scramble, 0));
  const float fy = fis_sample(fr.fis, samp2(fr, 1, s, scramble, 0));
  const float sx = ((float)x + 0.5f) + fx;
  const float sy = ((float)y + 0.5f) + fy;
  const float u = (1.0f / (float)fr.W) * sx;
  const float v = (1.0f / (float)fr.H) * sy;
  const float time = fr.t0 + (fr.t1 - fr.t0) * samp1(fr, s, scramble, 0);
  const float ls0 = samp2(fr, 0, s, scramble, 1), ls1 = samp2(fr, 1, s, scramble, 1);
  const float time0 = fr.t0 + (fr.t1 - fr.t0) * samp1(fr, s & ~3, scramble, 0);  // lane 0 of this sample's camera packet
  f3 ro, rd;
  camera_ray(sc.cam, u, v, ls0, ls1, time0, &ro, &rd);
  const size_t g = (size_t)ts * pb.R + i;
  float closest = 0.0f;
  int hit_id = -1;
  if (pre_n >= 0) fold_head(sc, pre_n, ro, rd, &closest, &hit_id);  // pre_n < 0: k_extend_spheres starts the fold (moving spheres)
  pb.o_time[g] = make_float4(ro.x, ro.y, ro.z, time);
  pb.d_t[g] = make_float4(rd.x, rd.y, rd.z, closest);
  pb.q_key[g] = hit_id;
  pb.rad[g] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  pb.thr[g] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
  pb.nrm0[g] = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(0u));
  pb.term[g] = 0u;
  pb.q_live[g] = i;
}
template __global__ void k_raygen<DevScene>(const __grid_constant__ DevScene, const DevFrame, const PassBufs, const int);

// ------------------------------------------------------------------------------------------
// K3 bin+pad: HitStore::add_hit / process_hits (hitable.rs:90-133).  Stable partition of a
// tile's live rays by object id, every bin padded to a multiple of 4 with -1.  One CTA per
// tile; chunks of BIN_T rays; per-warp __match_any_sync ranks + cross-warp offsets in smem.
// ------------------------------------------------------------------------------------------
#define BIN_T 1024
#define SEG_SLOTS 32768  // rays / slots one CTA of the per-tile queue kernels (bin, compact) walks
// Two kernels, grid (segments, tiles): at 4096 spp a tile holds 1 Mi rays and a pass only 96 tiles, so one CTA per tile
// (round 1 and 2a) left a third of the SMs idle and walked 1024 chunks serially - the 8-GPU weak-scaled config-3 run lost 5 %
// of its frame here.  A tile's live list is cut into SEG_SLOTS-ray segments; k_bin_count leaves per-segment per-object counts in
// HBM, k_bin_scatter turns them into the segment's write cursors and scatters.  The partition stays stable (segments are in
// order, a segment is scattered in order), so the queue is the same as the single-CTA one, bit for bit.
// MAXK = the scene type's kMaxHit: the number of keys, and the row stride of seg_cnt
template <int MAXK>
__global__ void __launch_bounds__(BIN_T) k_bin_count(const PassBufs pb, const int n_hit, const int nseg) {
  const int seg = blockIdx.x, ts = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
  const int n = pb.n_live[ts];
  __shared__ int cnt[MAXK];
  const int* __restrict__ qk = pb.q_key + (size_t)ts * pb.R;  // per path
  const int* __restrict__ ql = pb.q_live + (size_t)ts * pb.R;
  if (tid < MAXK) cnt[tid] = 0;
  if (tid == 0 && seg == 0 && n) atomicAdd(pb.counters + CNT_EXTEND_RAYS, (unsigned long long)n);  // rays through the closest-hit stage
  __syncthreads();
  const int lo = seg * SEG_SLOTS, hi = min(n, lo + SEG_SLOTS);
  for (int base = lo; base < hi; base += BIN_T) {
    const int i = base + tid;
    const int key = i < hi ? qk[ql[i]] : -1;
    const unsigned m = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && (m & ((1u << lane) - 1)) == 0) atomicAdd(&cnt[key], __popc(m));
  }
  __syncthreads();
  if (tid < n_hit) pb.seg_cnt[((size_t)ts * nseg + seg) * MAXK + tid] = cnt[tid];
}
template __global__ void k_bin_count<SCENE_INLINE_MAX>(const PassBufs, const int, const int);
__global__ void __launch_bounds__(BIN_T) k_bin_scatter(const PassBufs pb, const int n_hit, const int nseg) {
  const int seg = blockIdx.x, ts = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = BIN_T / 32;
  const int n = pb.n_live[ts];
  const int lo = seg * SEG_SLOTS, hi = min(n, lo + SEG_SLOTS);
  if (lo >= n && seg > 0) return;  // nothing to scatter; segment 0 still publishes the (possibly empty) bin table
  __shared__ int cnt[SCENE_INLINE_MAX];        // whole-tile counts
  __shared__ int before[SCENE_INLINE_MAX];     // counts of the segments before this one
  __shared__ int start[SCENE_INLINE_MAX + 1];
  __shared__ int running[2][SCENE_INLINE_MAX];
  __shared__ int wcnt[2][NW][SCENE_INLINE_MAX];
  const int* __restrict__ qk = pb.q_key + (size_t)ts * pb.R;
  const int* __restrict__ ql = pb.q_live + (size_t)ts * pb.R;
  int* __restrict__ qs = pb.q_shade + (size_t)ts * pb.QS;
  if (tid < n_hit) {
    const int used = (n + SEG_SLOTS - 1) / SEG_SLOTS;
    int tot = 0, bef = 0;
    for (int sg = 0; sg < used; ++sg) {
      const int c = pb.seg_cnt[((size_t)ts * nseg + sg) * SCENE_INLINE_MAX + tid];
      if (sg < seg) bef += c;
      tot += c;
    }
    cnt[tid] = tot, before[tid] = bef;
  }
  __syncthreads();
  if (tid == 0) {
    int off = 0;
    for (int o = 0; o < n_hit; ++o) {
      start[o] = off;
      running[0][o] = off + before[o];
      off += (cnt[o] + 3) & ~3;  // every bin padded to a multiple of 4 (hitable.rs:100-111)
    }
    start[n_hit] = off;
    if (seg == 0) pb.n_slots[ts] = off;
  }
  __syncthreads();
  if (seg == 0 && tid <= n_hit) pb.bin_start[ts * (SCENE_INLINE_MAX + 1) + tid] = start[tid];
  // stable scatter of this segment, ONE barrier per 1024-ray chunk (double-buffered warp counts and bin cursors)
  int buf = 0;
  for (int base = lo; base < hi; base += BIN_T, buf ^= 1) {
    const int i = base + tid;
    const int id = i < hi ? ql[i] : -1;
    const int key = i < hi ? qk[id] : -1;
    unsigned mine = 0;
    for (int k = 0; k < n_hit; ++k) {
      const unsigned b = __ballot_sync(0xffffffffu, key == k);
      if (key == k) mine = b;
      if (lane == k) wcnt[buf][warp][k] = __popc(b);
    }
    __syncthreads();
    if (key >= 0) {
      int off = running[buf][key] + __popc(mine & ((1u << lane) - 1));
      for (int w = 0; w < warp; ++w) off += wcnt[buf][w][key];
      qs[off] = id;
    }
    if (tid < n_hit) {
      int tot = running[buf][tid];
      for (int w = 0; w < NW; ++w) tot += wcnt[buf][w][tid];
      running[buf ^ 1][tid] = tot;
    }
  }
  if (seg == 0 && tid < n_hit)
    for (int k = start[tid] + cnt[tid]; k < start[tid + 1]; ++k) qs[k] = -1;  // Ray::new_invalid padding
}
// The same partition for scenes of up to RAYN_MAX_HITABLES keys (after k_bin_count<RAYN_MAX_HITABLES>).  k_bin_scatter's one
// ballot per key and chunk, and its [2][32][keys] warp counts (256 KB at 1024 keys), do not scale; here a warp ranks its rays
// with __match_any_sync (rank among the warp's rays of the same key), the leader of each key group posts the group's size
// in wcnt[warp][key], and a ray's slot is its bin cursor + the sizes posted by the warps before it + its rank.  A smaller
// CTA keeps wcnt at 8 x 4 KB; the leaders clear their entries after use, so no chunk pays for the keys it does not touch.
// Same order as k_bin_scatter: segments in order, chunks in order, warps in order, lanes in order.
#define BINB_T 256
__global__ void __launch_bounds__(BINB_T) k_bin_scatter_tables(const PassBufs pb, const int n_hit, const int nseg) {
  constexpr int K = RAYN_MAX_HITABLES, NW = BINB_T / 32, PER = K / BINB_T;
  static_assert(K % BINB_T == 0, "keys per thread of the bin scan");
  const int seg = blockIdx.x, ts = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt = (1u << lane) - 1u;
  const int n = pb.n_live[ts];
  const int lo = seg * SEG_SLOTS, hi = min(n, lo + SEG_SLOTS);
  if (lo >= n && seg > 0) return;
  __shared__ int cnt[K];        // whole-tile counts
  __shared__ int start[K + 1];  // bin starts (padded to x4)
  __shared__ int running[K];    // write cursor of every bin in this segment
  __shared__ int wcnt[NW][K];   // per-warp key counts of the current chunk, 0 where a warp has no such key
  __shared__ int wsum[NW];
  const int* __restrict__ qk = pb.q_key + (size_t)ts * pb.R;
  const int* __restrict__ ql = pb.q_live + (size_t)ts * pb.R;
  int* __restrict__ qs = pb.q_shade + (size_t)ts * pb.QS;
  const int used = (n + SEG_SLOTS - 1) / SEG_SLOTS;
  for (int k = tid; k < K; k += BINB_T) {
    int tot = 0, bef = 0;
    if (k < n_hit)
      for (int sg = 0; sg < used; ++sg) {
        const int c = pb.seg_cnt[((size_t)ts * nseg + sg) * K + k];
        if (sg < seg) bef += c;
        tot += c;
      }
    cnt[k] = tot, running[k] = bef;
#pragma unroll
    for (int w = 0; w < NW; ++w) wcnt[w][k] = 0;
  }
  __syncthreads();
  // exclusive scan of the padded bin sizes (hitable.rs:100-111): thread t owns keys PER*t .. PER*t + PER-1
  int sz[PER], s = 0;
#pragma unroll
  for (int q = 0; q < PER; ++q) s += (sz[q] = (cnt[PER * tid + q] + 3) & ~3);
  int x = s;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) wsum[warp] = x;
  __syncthreads();
  int off = x - s;
  for (int w = 0; w < warp; ++w) off += wsum[w];
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    start[PER * tid + q] = off;
    running[PER * tid + q] += off;
    off += sz[q];
  }
  if (tid == BINB_T - 1) start[K] = off;
  __syncthreads();
  if (seg == 0) {
    if (tid == 0) pb.n_slots[ts] = start[K];  // keys >= n_hit are empty: start[n_hit] == start[K]
    for (int k = tid; k <= n_hit; k += BINB_T) pb.bin_start[(size_t)ts * (K + 1) + k] = start[k];
  }
  for (int base = lo; base < hi; base += BINB_T) {
    const int i = base + tid;
    const int id = i < hi ? ql[i] : -1;
    const int key = i < hi ? qk[id] : -1;
    const unsigned m = __match_any_sync(0xffffffffu, key);
    const bool leader = key >= 0 && (m & lt) == 0;
    if (leader) wcnt[warp][key] = __popc(m);
    __syncthreads();
    if (key >= 0) {
      int o = running[key] + __popc(m & lt);
      for (int w = 0; w < warp; ++w) o += wcnt[w][key];
      qs[o] = id;
    }
    __syncthreads();
    if (leader) {
      atomicAdd(&running[key], __popc(m));  // read again only after the next chunk's first barrier
      wcnt[warp][key] = 0;
    }
    __syncwarp();  // the clear above is ordered before this warp's posts of the next chunk
  }
  if (seg == 0)
    for (int k = tid; k < n_hit; k += BINB_T)
      for (int j = start[k] + cnt[k]; j < start[k + 1]; ++j) qs[j] = -1;  // Ray::new_invalid padding
}

// ---- pass-wide work distribution for the persistent march kernels: the per-tile live lists are
// flattened into 128-ray batches numbered across the whole pass (k_scan_live builds the prefix) and
// resident warps pull batches from ONE global counter until the pass is drained, so the only tail
// is at the very end of the kernel (round-1 history of this design: DESIGN.md §4).
#define EXT_BATCH 128
#define SCAN_T 1024
__global__ void __launch_bounds__(SCAN_T) k_scan_live(const PassBufs pb, int* __restrict__ batch_prefix, int* __restrict__ work_ctr) {
  // batch_prefix[ts] = sum_{u<ts} ceil(n_live[u] / EXT_BATCH); batch_prefix[n_tiles] = total
  __shared__ int wsum[SCAN_T / 32];
  __shared__ int carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    carry = 0;
  }
  if (tid < WC_TOTAL) work_ctr[tid] = 0;  // extend batches, shadow batches and pushed-segment counts (PassBufs::seg_count)
  __syncthreads();
  for (int base = 0; base < pb.n_tiles; base += SCAN_T) {
    const int i = base + tid;
    const int v = i < pb.n_tiles ? (pb.n_live[i] + EXT_BATCH - 1) / EXT_BATCH : 0;
    int x = v;
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int w = wsum[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      wsum[lane] = w;
    }
    __syncthreads();
    const int excl = carry + (warp ? wsum[warp - 1] : 0) + x - v;
    if (i < pb.n_tiles) batch_prefix[i] = excl;
    __syncthreads();
    if (tid == SCAN_T - 1) carry = excl + v;
    __syncthreads();
  }
  if (tid == 0) batch_prefix[pb.n_tiles] = carry;
}

// Work lists of the slot-parallel kernels.  Round-2 launch list (profiles/r02_cfg3_launches.md): with a grid of
// (QS / 128, tiles) blocks k_normals / k_shade_pre / k_shade_post cost a constant 0.41 ms per launch at depths 4-8, where hardly
// a path is alive - 787 k empty blocks each, 5 % of a config-3 frame.  k_scan_slots (one CTA, after k_bin_scatter) lays the
// NON-EMPTY 128-slot blocks of all tiles end to end; the kernels run a resident grid that strides over that list.
#define SLOT_BLOCK 128
template <class Scn>
__global__ void __launch_bounds__(SCAN_T) k_scan_slots(const __grid_constant__ Scn sc, const PassBufs pb) {
  __shared__ int wsum[SCAN_T / 32];
  __shared__ int carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int row = 0; row <= sc.n_sdf; ++row) {
    int* __restrict__ out = pb.slot_prefix + (size_t)row * pb.prefix_stride;
    const int hk = row ? sc.sdf_idx[row - 1] : 0;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < pb.n_tiles; base += SCAN_T) {
      const int i = base + tid;
      int v = 0;
      if (i < pb.n_tiles) {
        const int* __restrict__ bs = pb.bin_start + i * (Scn::kMaxHit + 1);
        const int slots = row ? bs[hk + 1] - bs[hk] : pb.n_slots[i];
        v = (slots + SLOT_BLOCK - 1) / SLOT_BLOCK;
      }
      int x = v;
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) wsum[warp] = x;
      __syncthreads();
      if (warp == 0) {
        int w = wsum[lane];
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, w, o);
          if (lane >= o) w += y;
        }
        wsum[lane] = w;
      }
      __syncthreads();
      const int excl = carry + (warp ? wsum[warp - 1] : 0) + x - v;
      if (i < pb.n_tiles) out[i] = excl;
      __syncthreads();
      if (tid == SCAN_T - 1) carry = excl + v;
      __syncthreads();
    }
    if (tid == 0) out[pb.n_tiles] = carry;
    __syncthreads();
  }
}
template __global__ void k_scan_slots<DevScene>(const __grid_constant__ DevScene, const PassBufs);
// The resident CTAs of a work-list kernel pull WORK_CHUNK consecutive 128-slot blocks at a time from a global counter (zeroed
// by k_scan_live at the start of the depth).  Static striding was measured first: blocks differ 15x in cost (sky vs lit), the
// slowest CTA ran ~10 % over the mean and k_shade_pre lost more than the empty blocks had cost.
#define WORK_CHUNK 8
RT_D int grab_chunk(int* __restrict__ ctr, int* s_slot) {
  if (threadIdx.x == 0) *s_slot = atomicAdd(ctr, WORK_CHUNK);
  __syncthreads();
  const int c = *s_slot;
  __syncthreads();
  return c;
}
// work block wb of a prefix row -> tile slot whose blocks are [prefix[ts], prefix[ts + 1]) (every thread of the CTA runs the
// same search; the loads broadcast from L1)
RT_D int find_tile(const int* __restrict__ prefix, int n_tiles, int wb) {
  int lo = 0, hi = n_tiles;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(prefix + mid) <= wb) lo = mid; else hi = mid;
  }
  return lo;
}
// for (every work block wb of this CTA) BODY(ts, local)   with local = index of the block inside tile slot ts
#define FOR_EACH_WORK_BLOCK(prefix, n_tiles, ctr, ...)                                  \
  {                                                                                     \
    __shared__ int s_chunk_;                                                            \
    const int total_ = (prefix)[n_tiles];                                               \
    for (;;) {                                                                          \
      const int c0_ = grab_chunk(ctr, &s_chunk_);                                       \
      if (c0_ >= total_) break;                                                         \
      const int c1_ = min(c0_ + WORK_CHUNK, total_);                                    \
      int ts = 0, begin_ = 0, end_ = 0;                                                 \
      for (int wb_ = c0_; wb_ < c1_; ++wb_) {                                           \
        if (wb_ >= end_) {                                                              \
          ts = find_tile(prefix, n_tiles, wb_);                                         \
          begin_ = __ldg((prefix) + ts), end_ = __ldg((prefix) + ts + 1);               \
        }                                                                               \
        const int local = wb_ - begin_;                                                 \
        __VA_ARGS__                                                                     \
      }                                                                                 \
    }                                                                                   \
  }

// ---- K2 v4: closest hit split by hitable kind.  ncu on k_extend3 (profiles/r01 notes): the
// per-ray prologue/epilogue (sphere tests, gathers, stores) ran at 1-4 active lanes inside the
// persistent loop and cost more issue slots than the marches of cheap (sky) rays.  v4 keeps the
// fold order of hitable.rs:177-198 but runs every maximal run of analytic spheres as a coherent
// one-thread-per-ray kernel and every SDF hitable as a pure persistent march kernel.
template <class Scn>
__global__ void __launch_bounds__(EXT_BATCH) k_extend_spheres(const __grid_constant__ Scn sc, const PassBufs pb, const int first, const int last,
                                                              const int init, const int moving, const int* __restrict__ batch_prefix,
                                                              int* __restrict__ work_ctr) {
  // the 128-ray batches of k_scan_live: no block is launched for rays that are gone
  FOR_EACH_WORK_BLOCK(batch_prefix, pb.n_tiles, work_ctr, {
    const int i = local * EXT_BATCH + threadIdx.x;
    const int n = pb.n_live[ts];
    if (i < n) {
      const size_t q = (size_t)ts * pb.R + i;
      const size_t g = (size_t)ts * pb.R + pb.q_live[q];
      const float4 o4 = pb.o_time[g], d4 = pb.d_t[g];
      const f3 o = mk3(o4.x, o4.y, o4.z), d = mk3(d4.x, d4.y, d4.z);
      float closest = init ? sc.rc.world_radius * 2.0f : d4.w;  // film.rs:556
      int id = init ? -1 : pb.q_key[g];
      // packets of the extend stage are 4 consecutive live rays (film.rs:612-624); a moving sphere is evaluated at lane 0's time
      float time0 = o4.w;
      if (moving && (i & 3)) time0 = pb.o_time[(size_t)ts * pb.R + pb.q_live[(size_t)ts * pb.R + (i & ~3)]].w;
      for (int k = first; k < last; ++k) {
        const float t = moving ? sphere_hit(sc.hit[k], o, d, closest, time0) : sphere_hit_static(sc.sph[sc.hit_ord[k]], o, d, closest);
        if (t < closest) {
          closest = t;
          id = k;
        }
      }
      pb.d_t[g].w = closest;
      pb.q_key[g] = id;
    }
  })
}
template __global__ void k_extend_spheres<DevScene>(const __grid_constant__ DevScene, const PassBufs, const int, const int, const int, const int, const int*, int*);

// ------------------------------------------------------------------------------------------
// K2 sphere-march: TracedSDF::hit (sdf.rs:59-83, SURVEY §9.1) for SDF hitable `hk` over every live
// ray of the pass.  Persistent kernel: one wave of CTAs, warps pull 128-ray batches from a global
// counter.  Each THREAD marches TWO rays ("slots"); their state lives in float2 registers (component
// .x = slot 0, .y = slot 1) so the distance estimator runs on the packed f32x2 pipe (rt_sdf2.cuh).
// One loop trip = one distance evaluation on every busy slot of the warp; a slot whose march ended is
// refilled at the top of the next trip, so (nearly) all 64 slots of a warp evaluate every trip.  A march
// depends only on its own ray, so the order in which slots pick up work cannot change any output bit.
// The per-ray traffic is the algorithmic minimum: read float4 o+time, float4 d+closest (32 B), write
// t + key (8 B) when this SDF is the new closest hit.
//
// spheres_first != 0 (api.cu: fold_all): the producing kernel has already folded in EVERY analytic sphere, also those that
// follow this SDF in insertion order, and this march runs against the nearest of them.  That is the reference's fold
// (hitable.rs:177-198: in insertion order, strict `t < closest`, so the first index wins a tie) provided that
//  (1) a march's t never decreases - true for the Mandelbox, whose estimate sqrt(m) / |dr| is >= 0 or NaN - and
//  (2) a tie between this SDF and a sphere is resolved by index: the SDF wins exactly when the sphere comes later.
// Proof.  A sphere offers a candidate r* that does not depend on the bound it is tested against (sphere.rs:48-72: the bound only
// invalidates roots beyond it) and is accepted iff r* < closest, so the fold is a running strict minimum.  Let c0 be the minimum
// over the spheres before the SDF, c' <= c0 over all spheres.  The march visits the same t_0, t_1, ... whatever its bound;
// the bound only decides where it stops: the reference stops at the first i with (hit_i or t_i > c0), here at the first i'
// with (hit_i' or t_i' > c').  If i' = i both return the same T, and T wins the reference's fold iff T < c0 and T <= every later
// sphere's r*, which is `T < c'` or `T == c'` with c' owned by a later sphere.  If i' < i then c' < t_i' <= c0 (so c' belongs to
// a later sphere) and t_i' is rejected here; the reference marches on to T = t_i >= t_i' > c' by (1) (or to NaN), so that later
// sphere beats it there as well.  A NaN t is accepted by neither.
// ------------------------------------------------------------------------------------------
#define EXT_T 128
#ifndef RAYN_MARCH_OCC
#define RAYN_MARCH_OCC 8  // resident CTAs per SM the march kernels are compiled for (register budget 65536 / (128 * OCC))
#endif
#ifndef RAYN_MARCH_OCC_BULB
#define RAYN_MARCH_OCC_BULB RAYN_MARCH_OCC  // same for the authored Mandelbulb estimator (needs more registers; tuning hook)
#endif
#define MARCH_OCC(V) ((V) == SDFV_BULB ? RAYN_MARCH_OCC_BULB : RAYN_MARCH_OCC)
template <int V, class Scn>
__global__ void __launch_bounds__(EXT_T, MARCH_OCC(V)) k_extend_march(const __grid_constant__ Scn sc, const PassBufs pb, const Thr thr,
                                                          const int hk, const int spheres_first, const int* __restrict__ batch_prefix,
                                                          int* __restrict__ work_ctr) {
  const SdfK k = make_sdfk(sc.hit[hk], sc.one);  // fractal constants: kernel-parameter bank -> registers, once
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  const float S = sc.rc.sdf_detail_scale;
  const float c0 = 0.00005f * S, c1 = 0.05f * S;
  const bool c0_num = c0 == c0;  // max(c0, x) of the reference is NaN for a NaN c0: nothing ever "hits"
  const int max_marches = sc.rc.max_marches;
  const int n_batches = batch_prefix[pb.n_tiles];
  // slot state: g < 0 = empty; steps = -1 = the first evaluation (dist(origin), sdf.rs:60) is still to come.
  // Component .x of every packed value belongs to slot 0, .y to slot 1.
  pk2 ox = pk(0.0f, 0.0f), oy = ox, oz = ox, dx = ox, dy = ox, dz = ox;
  float2 t = splat2(0.0f), closest = t;
  int g0 = -1, g1 = -1, steps0 = -1, steps1 = -1, evals = 0, bulb_iters = 0, trips = 0;
  int cur_base = 0, cur_pos = 0, cur_end = 0;
  bool exhausted = false;
  while (true) {
    if (!exhausted || cur_pos < cur_end) {
      unsigned idle0 = __ballot_sync(0xffffffffu, g0 < 0), idle1 = __ballot_sync(0xffffffffu, g1 < 0);
      while (idle0 | idle1) {
        if (cur_pos >= cur_end) {
          int b = 0;
          if (lane == 0) b = atomicAdd(work_ctr, 1);
          b = __shfl_sync(0xffffffffu, b, 0);
          if (b >= n_batches) {
            exhausted = true;
            break;
          }
          int lo = 0, hi = pb.n_tiles;
          while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(batch_prefix + mid) <= b) lo = mid; else hi = mid;
          }
          cur_base = lo * pb.R;
          cur_pos = (b - __ldg(batch_prefix + lo)) * EXT_BATCH;
          cur_end = min(cur_pos + EXT_BATCH, pb.n_live[lo]);
        }
        const int avail = cur_end - cur_pos;
        const int n0 = __popc(idle0);
        const int rank0 = __popc(idle0 & lt), rank1 = n0 + __popc(idle1 & lt);
        if (g0 < 0 && rank0 < avail) {
          g0 = cur_base + pb.q_live[cur_base + cur_pos + rank0];
          const float4 o4 = pb.o_time[g0], d4 = pb.d_t[g0];
          ox = pk_set_x(ox, o4.x), oy = pk_set_x(oy, o4.y), oz = pk_set_x(oz, o4.z);
          dx = pk_set_x(dx, d4.x), dy = pk_set_x(dy, d4.y), dz = pk_set_x(dz, d4.z);
          closest.x = d4.w, t.x = 0.0f, steps0 = -1;
        }
        if (g1 < 0 && rank1 < avail) {
          g1 = cur_base + pb.q_live[cur_base + cur_pos + rank1];
          const float4 o4 = pb.o_time[g1], d4 = pb.d_t[g1];
          ox = pk_set_y(ox, o4.x), oy = pk_set_y(oy, o4.y), oz = pk_set_y(oz, o4.z);
          dx = pk_set_y(dx, d4.x), dy = pk_set_y(dy, d4.y), dz = pk_set_y(dz, d4.z);
          closest.y = d4.w, t.y = 0.0f, steps1 = -1;
        }
        cur_pos += min(avail, n0 + __popc(idle1));
        idle0 = __ballot_sync(0xffffffffu, g0 < 0), idle1 = __ballot_sync(0xffffffffu, g1 < 0);
      }
    }
    // while work remains every slot is busy here; slots stay empty only in the tail of the kernel, where they are parked on a
    // far point (cheapest for every estimator: the Mandelbulb leaves its loop at once and counts no iteration)
    if (exhausted) {
      if (!__any_sync(0xffffffffu, g0 >= 0 || g1 >= 0)) break;
      if (g0 < 0) ox = pk_set_x(ox, 100.0f), oy = pk_set_x(oy, 0.0f), oz = pk_set_x(oz, 0.0f), steps0 = -1;
      if (g1 < 0) ox = pk_set_y(ox, 100.0f), oy = pk_set_y(oy, 0.0f), oz = pk_set_y(oz, 0.0f), steps1 = -1;
    }
    // evaluation point of each slot: the origin for the first evaluation (sdf.rs:60), ray.point_at(t) afterwards
    // (ray.rs:22-24: dir.mul_add(t, origin))
    const bool first0 = steps0 < 0, first1 = steps1 < 0;
    const float2 o_x = un(ox), o_y = un(oy), o_z = un(oz);
    float2 px = muladd2(un(dx), t, o_x, k.one), py = muladd2(un(dy), t, o_y, k.one), pz = muladd2(un(dz), t, o_z, k.one);
    if (first0) px.x = o_x.x, py.x = o_y.x, pz.x = o_z.x;
    if (first1) px.y = o_x.y, py.y = o_y.y, pz.y = o_z.y;
    const float2 dd = sdf_dist2<V>(k, px, py, pz, bulb_iters);
    ++trips;
    // per-slot march step, branch-free up to the (rare) end of a march:
    //   first evaluation (sdf.rs:60-61): t = dist(origin), no hit test; a NaN start ends the march (the caller's t < closest is false);
    //   later (sdf.rs:65-80): stop on |dist| < max(0.00005 S, 0.05 S threshold(t)) or t > t_max, else t += dist; a NaN t can never
    //   satisfy hit/gt again, the reference marches it to exhaustion and returns NaN - ending at once returns the same NaN.
    //   max(c0, x) = (c0 < x ? x : c0): for a non-NaN c0, |d| < max(c0, x) <=> |d| < c0 || |d| < x  (x NaN: both sides |d| < c0).
    const float2 th = mul2(splat2(c1), thr.is_const ? splat2(thr.scale) : mul2(splat2(thr.scale), t));
    const float2 tsum = add2(t, dd);
    // (bitwise & | on the predicates: no short-circuit branches in the per-trip path)
    bool done0, done1, stop0, stop1;
    {
      const float ad = dm::abs(dd.x);
      stop0 = !first0 & ((c0_num & ((ad < c0) | (ad < th.x))) | (t.x > closest.x));
      const float tn = first0 ? dd.x : tsum.x;
      const int sn = steps0 + 1;
      t.x = stop0 ? t.x : tn;
      steps0 = stop0 ? steps0 : sn;
      done0 = stop0 | (tn != tn) | (sn >= max_marches);
    }
    {
      const float ad = dm::abs(dd.y);
      stop1 = !first1 & ((c0_num & ((ad < c0) | (ad < th.y))) | (t.y > closest.y));
      const float tn = first1 ? dd.y : tsum.y;
      const int sn = steps1 + 1;
      t.y = stop1 ? t.y : tn;
      steps1 = stop1 ? steps1 : sn;
      done1 = stop1 | (tn != tn) | (sn >= max_marches);
    }
    if (done0 | done1) {
      if (done0 & (g0 >= 0)) {
        if (t.x < closest.x || (spheres_first && t.x == closest.x && pb.q_key[g0] > hk)) {  // hitable.rs:190-193 (+ tie rule above)
          pb.d_t[g0].w = t.x;
          pb.q_key[g0] = hk;
        }
        evals += steps0 + (stop0 ? 2 : 1);  // distance evaluations this march took
        g0 = -1;
      }
      if (done1 & (g1 >= 0)) {
        if (t.y < closest.y || (spheres_first && t.y == closest.y && pb.q_key[g1] > hk)) {
          pb.d_t[g1].w = t.y;
          pb.q_key[g1] = hk;
        }
        evals += steps1 + (stop1 ? 2 : 1);
        g1 = -1;
      }
    }
  }
  warp_add(pb.counters + CNT_EVALS_EXTEND, evals);
  if (lane == 0) atomicAdd(pb.counters + CNT_TRIPS_EXTEND, (unsigned long long)trips);
  if (V == SDFV_BULB) warp_add(pb.counters + CNT_BULB_ITERS_EXTEND, bulb_iters);
}

// ------------------------------------------------------------------------------------------
// K3b normals: TracedSDF::get_shading_info (sdf.rs:85-101) for the shading slots of SDF hitable `hk`:
// sdfu's tetrahedral normals_fast (oracle/README.md A8) = 4 distance evaluations = 2 packed evaluations
// per lane, specialised on the SDF like the march kernels.  Writes nrm[g] = (normal, offset_by).
// ------------------------------------------------------------------------------------------
template <int V, class Scn>
__global__ void __launch_bounds__(128, 8) k_normals(const __grid_constant__ Scn sc, const PassBufs pb, const Thr thr, const int hk, const int j,
                                                    int* __restrict__ work_ctr) {
  const int* __restrict__ prefix = pb.slot_prefix + (size_t)(1 + j) * pb.prefix_stride;  // 128-slot blocks of this SDF's bins, all tiles
  const SdfK k = make_sdfk(sc.hit[hk], sc.one);
  int evals = 0;
  FOR_EACH_WORK_BLOCK(prefix, pb.n_tiles, work_ctr, {
    const int* __restrict__ bs = pb.bin_start + ts * (Scn::kMaxHit + 1);
    const int s = bs[hk] + local * SLOT_BLOCK + threadIdx.x;
    const int id = s < bs[hk + 1] ? pb.q_shade[(size_t)ts * pb.QS + s] : -1;
    if (id >= 0) {  // < 0: beyond the bin, or a padding lane (hitable.rs:100-111)
      const size_t g = (size_t)ts * pb.R + id;
      const float4 o4 = pb.o_time[g], d4 = pb.d_t[g];
      const f3 point = fma3s(mk3(d4.x, d4.y, d4.z), d4.w, mk3(o4.x, o4.y, o4.z));  // WHit::point -> ray.point_at, ray.rs:22-24
      const float eps = dm::max(0.0001f, sc.rc.sdf_detail_scale * thr.at(d4.w));
      // tetrahedron offsets k0 = (1,-1,-1), k1 = (-1,-1,1), k2 = (-1,1,-1), k3 = (1,1,1); n = ((k0 d0 + k1 d1) + k2 d2) + k3 d3
      int it = 0;
      const float ex = 1.0f * eps, en = -1.0f * eps;
      const float2 da = sdf_dist2<V>(k, f2(point.x + ex, point.x + en), f2(point.y + en, point.y + en), f2(point.z + en, point.z + ex), it);
      const float2 db = sdf_dist2<V>(k, f2(point.x + en, point.x + ex), f2(point.y + ex, point.y + ex), f2(point.z + en, point.z + ex), it);
      f3 n = mk3(1.0f, -1.0f, -1.0f) * da.x;
      n = n + mk3(-1.0f, -1.0f, 1.0f) * da.y;
      n = n + mk3(-1.0f, 1.0f, -1.0f) * db.x;
      n = n + mk3(1.0f, 1.0f, 1.0f) * db.y;
      n = normalized(n);
      pb.nrm[g] = make_float4(n.x, n.y, n.z, eps);
      evals += 4;
    }
  })
  warp_add(pb.counters + CNT_EVALS_NORMALS, evals);
}
// ==========================================================================================
// v3 shading: k_shade_pre -> k_shadow (persistent) -> k_shade_post.
// The block-level pool of k_shade2 still drains to a tail every round; v3 pushes the shadow
// segments of the whole pass into one HBM queue and marches it with resident warps that pull
// 64-segment batches from a global counter.  pre evaluates light_contrib() once per light sample and
// stores the unoccluded contribution (c.xyz, pdf [, transmission]) per path; post multiplies by the
// visibility bit and accumulates in the reference's order (HBM is idle here, ALU issue is not).
// ==========================================================================================
struct LightContrib {
  f3 start, end_point, c;
  float den, trans;
};
// round 0: surface_sample_one_light (integrator.rs:207-240) without the visibility factor;
// round r>0: volume_sample_one_light (:242-281) for volume march r-1.
RT_D LightContrib light_contrib(const RaynLight& L, const RaynMaterial& mat, const ShadingPoint& sp, f3 wo, int round, float u0, float u1,
                                float vol_sample, bool has_ext, float neg_rho_t) {
  LightContrib r;
  f3 li;
  r.trans = 1.0f;
  if (round == 0) {
    float pdf;
    light_sample(L, u0, u1, sp.point, &r.end_point, &li, &pdf);
    f3 wi = r.end_point - sp.point;
    const float dist = mag(wi);
    wi = wi / dist;
    r.start = sp.point + sp.normal * dm::signum(dot(sp.normal, wi)) * sp.offset_by;
    const f3 f = bsdf_f(mat, wo, wi, sp.normal) * dm::max(dot(sp.normal, wi), 0.0f);
    const float tr = has_ext ? dm::exp(neg_rho_t * dist) : 1.0f;
    r.c = li * f * tr;
    r.den = pdf;
  } else {
    float vol_dist, vol_pdf, light_pdf;
    light_sample_volume(L, vol_sample, sp.o, sp.d, sp.t, &vol_dist, &vol_pdf);
    r.start = sp.o + sp.d * vol_dist;
    light_sample(L, u0, u1, r.start, &r.end_point, &li, &light_pdf);
    const float dist_point_to_light = mag(r.end_point - r.start);
    const float f = 1.0f / (4.0f * RT_PI);
    const float tr = has_ext ? dm::exp(neg_rho_t * dist_point_to_light) : 1.0f;
    r.c = li * f * tr;
    r.den = vol_pdf * light_pdf;
    r.trans = has_ext ? dm::exp(neg_rho_t * vol_dist) : 1.0f;  // :122-126
  }
  return r;
}

struct SlotCtx {  // what pre and post both derive for a shading slot
  int id, sample, obj;
  float scramble;
  unsigned w0, w1, w2;  // light indices of the packet, one byte per packet lane, per round
  int set1, set2;
};
// Memory-level parallelism matters here (r02a profile: both shade kernels sit on long-scoreboard stalls at ~23 % issue
// utilisation): everything a slot needs hangs off ONE dependent load, its path id, so that the hit object (q_key is indexed
// by path), the pixel's scramble value and the sampler-table entries are all in flight together - the former search of the
// tile's bin_start row was a chain of up to n_hit dependent loads.
template <class Scn>
RT_D SlotCtx slot_ctx(const Scn& sc, const DevFrame& fr, const PassBufs& pb, int ts, int s, int nslots, int depth, int lane) {
  SlotCtx c;
  const int* __restrict__ qs = pb.q_shade + (size_t)ts * pb.QS;
  c.id = s < nslots ? qs[s] : -1;
  c.sample = 0;
  c.obj = 0;
  c.scramble = 0.0f;  // padded lanes are Ray::new_invalid: sample 0, scramble 0 (ray.rs:54-66)
  if (c.id >= 0) {
    c.obj = pb.q_key[(size_t)ts * pb.R + c.id];  // the bin this slot sits in (k_bin partitions by this key)
    const TileGeom tg = tile_geom(fr, pb.tile_ids[ts]);
    const int pl = c.id / fr.spp;
    c.sample = c.id - pl * fr.spp;
    const int xl = pl / tg.th, yl = pl - xl * tg.th;
    c.scramble = __ldg(fr.scramble + (tg.x0 + xl) + (size_t)(tg.y0 + yl) * fr.W);
  }
  const int n1 = 3 + fr.vm, n2h = (12 + 8 * fr.vm) / 2;
  c.set1 = 1 + depth * n1;
  c.set2 = 2 + depth * n2h;
  const int nl = sc.n_lights;
  unsigned pack = 0;
  if (nl > 0) {
    const float u0 = __ldg(fr.s1 + c.sample + (size_t)fr.spp * (c.set1 + 0)), u1 = __ldg(fr.s1 + c.sample + (size_t)fr.spp * (c.set1 + 1)),
                u2 = __ldg(fr.s1 + c.sample + (size_t)fr.spp * (c.set1 + 2));  // three independent loads, then samp1's fract(x + scramble)
    pack = (unsigned)light_index(dm::fract(u0 + c.scramble), nl) | ((unsigned)light_index(dm::fract(u1 + c.scramble), nl) << 8) |
           ((unsigned)light_index(dm::fract(u2 + c.scramble), nl) << 16);
  }
  c.w0 = c.w1 = c.w2 = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const unsigned pk = __shfl_sync(0xffffffffu, pack, (lane & ~3) + k);
    c.w0 |= (pk & 0xffu) << (8 * k);
    c.w1 |= ((pk >> 8) & 0xffu) << (8 * k);
    c.w2 |= ((pk >> 16) & 0xffu) << (8 * k);
  }
  return c;
}

template <class Scn>
RT_D void shade_pre_slot(const Scn& sc, const DevFrame& fr, const PassBufs& pb, const int depth, const Thr thr, const int ts, const int s) {
  const int nslots = pb.n_slots[ts];
  if ((s & ~31) >= nslots) return;  // warp-uniform
  const SlotCtx cx = slot_ctx(sc, fr, pb, ts, s, nslots, depth, threadIdx.x & 31);
  const bool valid = cx.id >= 0;
  warp_add(pb.counters + CNT_SHADE_LANES, valid ? 1 : 0);
  int shadows = 0;
  const size_t g = (size_t)ts * pb.R + (valid ? cx.id : 0);
  float4 o4 = make_float4(0, 0, 0, 0), d4 = o4, r4 = o4, t4 = o4;
  if (valid) o4 = pb.o_time[g], d4 = pb.d_t[g], r4 = pb.rad[g], t4 = pb.thr[g];  // all in flight before the shuffle below waits for o4
  // time of lane 0 of this shading packet (bins pad at the tail, so lane 0 of a non-empty packet is valid): what a
  // closure-backed Sphere centre is evaluated at in occluded() / get_shading_info() (sphere.rs:29,80; animation.rs:62-67)
  const float time0 = __shfl_sync(0xffffffffu, o4.w, (threadIdx.x & 31) & ~3);
  if (valid) {
    const RaynHitable& h = sc.hit[cx.obj];
    const RaynMaterial& mat = sc.mat[h.material];
    ShadingPoint sp;
    sp.o = mk3(o4.x, o4.y, o4.z);
    sp.d = mk3(d4.x, d4.y, d4.z);
    sp.time = o4.w;
    sp.t = d4.w;
    const bool recv = receives_light(mat);
    const int nl = sc.n_lights;
    const bool scat = sc.vol.has_scattering != 0 && nl > 0;
    const int n_rounds = nl > 0 ? 1 + (scat ? fr.vm : 0) : 0;
    const f3 wo = -sp.d;
    const bool has_ext = sc.vol.has_extinction != 0;
    const float neg_rho_t = -sc.vol.coeff_extinction;
    const float vt = has_ext ? dm::exp(neg_rho_t * sp.t) : 1.0f;  // integrator.rs:64-68
    const f3 radiance = mk3(r4.x, r4.y, r4.z) + bsdf_le(mat, wo) * mk3(t4.x, t4.y, t4.z) * vt;  // :70-71
    pb.rad[g] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
    if (!recv && !scat) {
      // Sky / Emissive without volumetrics: emission is the whole shading step (integrator.rs:70-71,
      // 189-203); the path ends here.  Every lane of its packet has the same material, so nobody needs
      // this lane's light choice and k_shade_post can treat the slot as empty.
      pb.term[g] = ((depth == 0 ? TERM_BACKGROUND : TERM_COLOR) << 30) | ((unsigned)depth << TERM_DEPTH_SHIFT) | (unsigned)s;
      pb.q_shade[(size_t)ts * pb.QS + s] = -1;
    } else {
      sp.point = fma3s(sp.d, sp.t, sp.o);  // WHit::point -> ray.point_at, ray.rs:22-24
      if (h.kind == RAYN_HITABLE_SPHERE) {  // sphere.rs:74-86
        sp.normal = normalized(sp.point - sphere_center(h, time0));
        sp.offset_by = 0.0f;
        pb.nrm[g] = make_float4(sp.normal.x, sp.normal.y, sp.normal.z, 0.0f);
      } else {  // sdf.rs:85-101: written by k_normals<V> for this hitable
        const float4 n4 = pb.nrm[g];
        sp.normal = mk3(n4.x, n4.y, n4.z);
        sp.offset_by = n4.w;
      }
      unsigned vis = 0xffffffffu;
      for (int round = (recv ? 0 : 1); round < n_rounds; ++round) {
        const unsigned wr = round == 0 ? cx.w0 : (round == 1 ? cx.w1 : cx.w2);
        const float vol_sample = round == 0 ? 0.0f : samp1(fr, cx.sample, cx.scramble, cx.set1 + 1);  // samples_1d[1], :115
#pragma unroll 1
        for (int i = 0; i < 4; ++i) {
          const int set = round == 0 ? cx.set2 + i : cx.set2 + 4 + 4 * (round - 1) + i;
          const LightContrib lc = light_contrib(sc.light[(wr >> (8 * i)) & 0xffu], mat, sp, wo, round, samp2(fr, 0, cx.sample, cx.scramble, set),
                                                samp2(fr, 1, cx.sample, cx.scramble, set), vol_sample, has_ext, neg_rho_t);
          ++shadows;
          const int bit = round * 4 + i;
          pb.lc_c[g * pb.lc_ns + bit] = make_float4(lc.c.x, lc.c.y, lc.c.z, lc.den);  // k_shade_post folds these in; HBM is idle, ALU is not
          if (round > 0) pb.lc_t[g * 8 + (bit - 4)] = lc.trans;
          // a contribution that is (+-0 | NaN) in every channel is the same bits for visibility 0 and 1
          const bool irrelevant = (lc.c.x == 0.0f || lc.c.x != lc.c.x) && (lc.c.y == 0.0f || lc.c.y != lc.c.y) && (lc.c.z == 0.0f || lc.c.z != lc.c.z);
          if (irrelevant) continue;
          // direction and length of the segment: the first three lines of every Hitable::occluded (sphere.rs:25-27, sdf.rs:26-28)
          f3 dir = lc.end_point - lc.start;
          const float max_dist = mag(dir);
          dir = dir / max_dist;
          float v = 1.0f;  // analytic spheres first, in insertion order: product of {0,1} factors (hitable.rs:164-168)
          if (sc.sph_moving) {
            for (int k = 0; k < sc.n_sph && v != 0.0f; ++k) v = sphere_occluded_seg(sc.hit[sc.sph_idx[k]], lc.start, dir, max_dist, time0);
          } else {
            for (int k = 0; k < sc.n_sph && v != 0.0f; ++k) v = sphere_occluded_seg_static(sc.sph[k], lc.start, dir, max_dist);
          }
          if (v == 0.0f) {
            vis &= ~(1u << bit);
            continue;
          }
          for (int j = 0; j < sc.n_sdf; ++j) {  // one shadow-segment queue per SDF hitable (ordinal j)
            const unsigned am = __activemask();  // opportunistic warp aggregation of the queue append
            const int leader = __ffs(am) - 1, ln = threadIdx.x & 31;
            int base = 0;
            if (ln == leader) base = atomicAdd(pb.seg_count + j, __popc(am));
            base = __shfl_sync(am, base, leader);
            const size_t slot = (size_t)j * pb.seg_cap + base + __popc(am & ((1u << ln) - 1u));
            pb.seg_a[slot] = make_float4(lc.start.x, lc.start.y, lc.start.z, max_dist);
            pb.seg_b[slot] = make_float4(dir.x, dir.y, dir.z, __int_as_float((int)(((unsigned)g << 4) | (unsigned)bit)));
          }
        }
      }
      pb.vis[g] = vis;
    }
  }
  warp_add(pb.counters + CNT_SHADOW_RAYS, shadows);
}

#ifndef RAYN_SHADE_PRE_OCC
#define RAYN_SHADE_PRE_OCC 8  // resident CTAs per SM k_shade_pre is compiled for (tuning hook)
#endif
template <class Scn>
__global__ void __launch_bounds__(128, RAYN_SHADE_PRE_OCC) k_shade_pre(const __grid_constant__ Scn sc, const DevFrame fr, const PassBufs pb,
                                                      const int depth, const Thr thr, int* __restrict__ work_ctr) {
  // row 0 of the work lists: the non-empty 128-slot blocks of every tile's shading queue
  FOR_EACH_WORK_BLOCK(pb.slot_prefix, pb.n_tiles, work_ctr, { shade_pre_slot(sc, fr, pb, depth, thr, ts, local * SLOT_BLOCK + threadIdx.x); })
}
template __global__ void k_shade_pre<DevScene>(const __grid_constant__ DevScene, const DevFrame, const PassBufs, const int, const Thr, int*);

// ------------------------------------------------------------------------------------------
// K5 shadow sphere-march: TracedSDF::occluded per slot (sdf.rs:25-57, SURVEY §9.2) over the segment
// queue of SDF ordinal `j` (hitable index `hk`); occlusion clears the owner's visibility bit.  Same
// persistent, two-slots-per-thread, packed-f32x2 structure as k_extend_march.  Traffic per segment:
// 32 B read (+ 4 B atomic when occluded).
// ------------------------------------------------------------------------------------------
#define SHD_T 128
#define SHD_BATCH 128
template <int V, class Scn>
__global__ void __launch_bounds__(SHD_T, MARCH_OCC(V)) k_shadow(const __grid_constant__ Scn sc, const PassBufs pb, const int hk, const int j,
                                                    int* __restrict__ work_ctr) {
  const SdfK k = make_sdfk(sc.hit[hk], sc.one);
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  const int n_seg = pb.seg_count[j];
  const float4* __restrict__ seg_a = pb.seg_a + (size_t)j * pb.seg_cap;
  const float4* __restrict__ seg_b = pb.seg_b + (size_t)j * pb.seg_cap;
  const float S = sc.rc.sdf_detail_scale;
  const float oc0 = 0.0001f * S, oc1 = 0.00001f * S;
  const bool oc0_num = oc0 == oc0;  // see k_extend_march
  const int max_vis = sc.rc.max_vis_marches;
  // slot state (see k_extend_march): own < 0 = empty, steps = -1 = dist(start) (sdf.rs:30) still to come
  pk2 sx = pk(0.0f, 0.0f), sy = sx, sz = sx, dx = sx, dy = sx, dz = sx;
  float2 t = splat2(0.0f), max_dist = t;
  int own0 = -1, own1 = -1, steps0 = -1, steps1 = -1, evals = 0, bulb_iters = 0, trips = 0;
  int cur_pos = 0, cur_end = 0;
  bool exhausted = false;
  while (true) {
    if (!exhausted || cur_pos < cur_end) {
      unsigned idle0 = __ballot_sync(0xffffffffu, own0 < 0), idle1 = __ballot_sync(0xffffffffu, own1 < 0);
      while (idle0 | idle1) {
        if (cur_pos >= cur_end) {
          int b = 0;
          if (lane == 0) b = atomicAdd(work_ctr, SHD_BATCH);
          b = __shfl_sync(0xffffffffu, b, 0);
          if (b >= n_seg) {
            exhausted = true;
            break;
          }
          cur_pos = b;
          cur_end = min(b + SHD_BATCH, n_seg);
        }
        const int avail = cur_end - cur_pos;
        const int n0 = __popc(idle0);
        const int rank0 = __popc(idle0 & lt), rank1 = n0 + __popc(idle1 & lt);
        if (own0 < 0 && rank0 < avail) {
          const float4 a = seg_a[cur_pos + rank0], b4 = seg_b[cur_pos + rank0];
          sx = pk_set_x(sx, a.x), sy = pk_set_x(sy, a.y), sz = pk_set_x(sz, a.z);
          dx = pk_set_x(dx, b4.x), dy = pk_set_x(dy, b4.y), dz = pk_set_x(dz, b4.z);
          max_dist.x = a.w, t.x = 0.0f, steps0 = -1;
          own0 = __float_as_int(b4.w);
        }
        if (own1 < 0 && rank1 < avail) {
          const float4 a = seg_a[cur_pos + rank1], b4 = seg_b[cur_pos + rank1];
          sx = pk_set_y(sx, a.x), sy = pk_set_y(sy, a.y), sz = pk_set_y(sz, a.z);
          dx = pk_set_y(dx, b4.x), dy = pk_set_y(dy, b4.y), dz = pk_set_y(dz, b4.z);
          max_dist.y = a.w, t.y = 0.0f, steps1 = -1;
          own1 = __float_as_int(b4.w);
        }
        cur_pos += min(avail, n0 + __popc(idle1));
        idle0 = __ballot_sync(0xffffffffu, own0 < 0), idle1 = __ballot_sync(0xffffffffu, own1 < 0);
      }
    }
    if (exhausted) {  // tail of the kernel: empty slots are parked on a far point (see k_extend_march)
      if (!__any_sync(0xffffffffu, own0 >= 0 || own1 >= 0)) break;
      if (own0 < 0) sx = pk_set_x(sx, 100.0f), sy = pk_set_x(sy, 0.0f), sz = pk_set_x(sz, 0.0f), steps0 = -1;
      if (own1 < 0) sx = pk_set_y(sx, 100.0f), sy = pk_set_y(sy, 0.0f), sz = pk_set_y(sz, 0.0f), steps1 = -1;
    }
    const bool first0 = steps0 < 0, first1 = steps1 < 0;
    const float2 s_x = un(sx), s_y = un(sy), s_z = un(sz);
    float2 px = muladd2(un(dx), t, s_x, k.one), py = muladd2(un(dy), t, s_y, k.one), pz = muladd2(un(dz), t, s_z, k.one);  // dir.mul_add(t, start), sdf.rs:45
    if (first0) px.x = s_x.x, py.x = s_y.x, pz.x = s_z.x;                                                                  // dist(start), sdf.rs:30
    if (first1) px.y = s_x.y, py.y = s_y.y, pz.y = s_z.y;
    const float2 dd = sdf_dist2<V>(k, px, py, pz, bulb_iters);
    ++trips;
    // per-slot step of TracedSDF::occluded, branch-free up to the end of a march (see k_extend_march):
    //   first (sdf.rs:30-36): t = dist(start);   later (:40-55): occluded when |dist| < max(1e-4 S, 1e-5 S t), else t += dist;
    //   the march ends unoccluded when t is NaN, exceeds max_dist, or after MAX_VIS_MARCHES steps.
    const float2 th = mul2(splat2(oc1), t);
    const float2 tsum = add2(t, dd);
    bool done0, done1, occ0, occ1;
    {
      const float ad = dm::abs(dd.x);
      occ0 = !first0 & oc0_num & ((ad < oc0) | (ad < th.x));
      const float tn = first0 ? dd.x : tsum.x;
      t.x = tn;
      steps0 = steps0 + 1;
      done0 = occ0 | (tn != tn) | (steps0 >= max_vis) | (tn > max_dist.x);
    }
    {
      const float ad = dm::abs(dd.y);
      occ1 = !first1 & oc0_num & ((ad < oc0) | (ad < th.y));
      const float tn = first1 ? dd.y : tsum.y;
      t.y = tn;
      steps1 = steps1 + 1;
      done1 = occ1 | (tn != tn) | (steps1 >= max_vis) | (tn > max_dist.y);
    }
    if (done0 | done1) {
      if (done0 & (own0 >= 0)) {
        if (occ0) atomicAnd(pb.vis + ((unsigned)own0 >> 4), ~(1u << (own0 & 15)));
        evals += steps0 + 1;  // distance evaluations this march took
        own0 = -1;
      }
      if (done1 & (own1 >= 0)) {
        if (occ1) atomicAnd(pb.vis + ((unsigned)own1 >> 4), ~(1u << (own1 & 15)));
        evals += steps1 + 1;
        own1 = -1;
      }
    }
  }
  warp_add(pb.counters + CNT_EVALS_SHADOW, evals);
  if (lane == 0) atomicAdd(pb.counters + CNT_TRIPS_SHADOW, (unsigned long long)trips);
  if (V == SDFV_BULB) warp_add(pb.counters + CNT_BULB_ITERS_SHADOW, bulb_iters);
}

template <class Scn>
RT_D void shade_post_slot(const Scn& sc, const DevFrame& fr, const PassBufs& pb, const int depth, const int pre_n, const int ts, const int s) {
  const int nslots = pb.n_slots[ts];
  if ((s & ~31) >= nslots) return;
  const SlotCtx cx = slot_ctx(sc, fr, pb, ts, s, nslots, depth, threadIdx.x & 31);
  if (cx.id < 0) return;
  int* __restrict__ qs = pb.q_shade + (size_t)ts * pb.QS;
  const RaynHitable& h = sc.hit[cx.obj];
  const RaynMaterial& mat = sc.mat[h.material];
  const size_t g = (size_t)ts * pb.R + cx.id;
  const float4 o4 = pb.o_time[g], d4 = pb.d_t[g], r4 = pb.rad[g], t4 = pb.thr[g], n4 = pb.nrm[g];
  ShadingPoint sp;
  sp.o = mk3(o4.x, o4.y, o4.z);
  sp.d = mk3(d4.x, d4.y, d4.z);
  sp.time = o4.w;
  sp.t = d4.w;
  sp.point = fma3s(sp.d, sp.t, sp.o);
  sp.normal = mk3(n4.x, n4.y, n4.z);
  sp.offset_by = n4.w;
  sp.basis = onb(sp.normal);
  f3 radiance = mk3(r4.x, r4.y, r4.z), throughput = mk3(t4.x, t4.y, t4.z);
  const f3 wo = -sp.d;
  const bool has_ext = sc.vol.has_extinction != 0;
  const float neg_rho_t = -sc.vol.coeff_extinction;
  const float vt = has_ext ? dm::exp(neg_rho_t * sp.t) : 1.0f;
  const bool recv = receives_light(mat);
  const int nl = sc.n_lights;
  const bool scat = sc.vol.has_scattering != 0 && nl > 0;
  const int n_rounds = nl > 0 ? 1 + (scat ? fr.vm : 0) : 0;
  const unsigned vis = pb.vis[g];
  for (int round = (recv ? 0 : 1); round < n_rounds; ++round) {
    const float correction = round == 0 ? (float)nl / 4.0f : (float)nl / 4.0f / (float)fr.vm;  // :79-80,104-108
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int bit = round * 4 + i;
      const float4 c4 = pb.lc_c[g * pb.lc_ns + bit];  // li * f * transmission and pdf, written by k_shade_pre
      const float occluded = (vis >> bit) & 1u ? 1.0f : 0.0f;
      // :239 / :278 `li * f * occluded / pdf`.  An occluded or back-facing sample has a (+-0, +-0, +-0) numerator, and +-0 / pdf is
      // that same +-0 for every pdf > 0: no division then (r02c profile: zero numerators send IEEE division down its slow
      // path, 17 % of this kernel's instructions).  NaN numerators and pdf <= 0 / NaN take the division as before.
      const f3 num = mk3(c4.x, c4.y, c4.z) * occluded;
      const bool no_div = (num.x == 0.0f) & (num.y == 0.0f) & (num.z == 0.0f) & (c4.w > 0.0f);
      const f3 contrib = no_div ? num : num / c4.w;
      if (round == 0)
        radiance = radiance + contrib * throughput * correction * vt;  // :91-92
      else
        radiance = radiance + contrib * throughput * correction * sc.vol.coeff_scattering * pb.lc_t[g * 8 + (bit - 4)];  // :128-129
    }
  }
  if (recv) {  // :134-188
    const int setb = cx.set2 + 4 + 4 * fr.vm;
    const Scatter se = bsdf_scatter(mat, wo, sp, samp1(fr, cx.sample, cx.scramble, cx.set1 + 3), samp2(fr, 0, cx.sample, cx.scramble, setb),
                                    samp2(fr, 1, cx.sample, cx.scramble, setb), samp2(fr, 0, cx.sample, cx.scramble, setb + 1),
                                    samp2(fr, 1, cx.sample, cx.scramble, setb + 1));
    const float ndl = dm::abs(dot(se.wi, sp.normal));
    f3 new_throughput = throughput * vt * se.f * ndl / se.pdf;
    float roulette_factor = 0.0f;
    if (depth > 2) {
      roulette_factor = dm::max(1.0f - component_max(throughput), 0.05f);
      new_throughput = new_throughput / (1.0f - roulette_factor);
    }
    if (depth == 0) pb.nrm0[g] = make_float4(sp.normal.x, sp.normal.y, sp.normal.z, __uint_as_float((unsigned)s + 1u));
    const float roulette_sample = samp1(fr, cx.sample, cx.scramble, cx.set1 + 4);
    if (depth >= fr.max_bounces || roulette_sample < roulette_factor) {
      pb.rad[g] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
      pb.term[g] = (TERM_COLOR << 30) | ((unsigned)depth << TERM_DEPTH_SHIFT) | (unsigned)s;
      qs[s] = -1;
    } else {
      const f3 no = sp.point + sp.normal * dm::signum(dot(sp.normal, se.wi)) * sp.offset_by;
      if (!any_nan(new_throughput)) throughput = new_throughput;
      float closest = 0.0f;
      int hit_id = -1;
      if (pre_n >= 0) fold_head(sc, pre_n, no, se.wi, &closest, &hit_id);  // head of the next depth's closest-hit fold
      pb.o_time[g] = make_float4(no.x, no.y, no.z, sp.time);
      pb.d_t[g] = make_float4(se.wi.x, se.wi.y, se.wi.z, closest);
      pb.q_key[g] = hit_id;
      pb.rad[g] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
      pb.thr[g] = make_float4(throughput.x, throughput.y, throughput.z, 0.0f);
    }
  } else {  // :189-203
    pb.rad[g] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
    pb.term[g] = ((depth == 0 ? TERM_BACKGROUND : TERM_COLOR) << 30) | ((unsigned)depth << TERM_DEPTH_SHIFT) | (unsigned)s;
    qs[s] = -1;
  }
}

template <class Scn>
__global__ void __launch_bounds__(128, 8) k_shade_post(const __grid_constant__ Scn sc, const DevFrame fr, const PassBufs pb,
                                                       const int depth, const int pre_n, int* __restrict__ work_ctr) {
  FOR_EACH_WORK_BLOCK(pb.slot_prefix, pb.n_tiles, work_ctr, { shade_post_slot(sc, fr, pb, depth, pre_n, ts, local * SLOT_BLOCK + threadIdx.x); })
}
template __global__ void k_shade_post<DevScene>(const __grid_constant__ DevScene, const DevFrame, const PassBufs, const int, const int, int*);

// ------------------------------------------------------------------------------------------
// K6 compact: film.rs:604-625.  Order-preserving stream compaction of the surviving slots of
// a tile into the next live queue: per-warp __ballot_sync + popc prefix, cross-warp offsets
// in shared memory, running tile offset.  (Padding the survivors to x4, film.rs:608-610, has
// no observable effect: add_hits drops invalid lanes, hitable.rs:204.)
// ------------------------------------------------------------------------------------------
#define CMP_T 1024
// grid (segments, tiles) like k_bin_*: survivors per SEG_SLOTS-slot segment, then every segment writes at the sum of the counts
// before it - the same order-preserving compaction as one CTA walking the whole tile.
__global__ void __launch_bounds__(CMP_T) k_compact_count(const PassBufs pb, const int nseg) {
  const int seg = blockIdx.x, ts = blockIdx.y, tid = threadIdx.x;
  const int n = pb.n_slots[ts];
  const int* __restrict__ qs = pb.q_shade + (size_t)ts * pb.QS;
  const int lo = seg * SEG_SLOTS, hi = min(n, lo + SEG_SLOTS);
  int c = 0;
  for (int i = lo + tid; i < hi; i += CMP_T) c += qs[i] >= 0 ? 1 : 0;
  c = __reduce_add_sync(0xffffffffu, c);
  __shared__ int tot;
  if (tid == 0) tot = 0;
  __syncthreads();
  if ((tid & 31) == 0 && c) atomicAdd(&tot, c);
  __syncthreads();
  if (tid == 0) pb.seg_cnt[((size_t)ts * nseg + seg) * SCENE_INLINE_MAX] = tot;
}
__global__ void __launch_bounds__(CMP_T) k_compact_scatter(const PassBufs pb, const int nseg) {
  const int seg = blockIdx.x, ts = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = CMP_T / 32;
  const int n = pb.n_slots[ts];
  const int lo = seg * SEG_SLOTS, hi = min(n, lo + SEG_SLOTS);
  if (lo >= n && seg > 0) return;
  const int* __restrict__ qs = pb.q_shade + (size_t)ts * pb.QS;
  int* __restrict__ ql = pb.q_live + (size_t)ts * pb.R;
  __shared__ int wtot[2][NW];
  __shared__ int running[2];
  if (tid == 0) {
    const int used = (n + SEG_SLOTS - 1) / SEG_SLOTS;
    int bef = 0, tot = 0;
    for (int sg = 0; sg < used; ++sg) {
      const int c = pb.seg_cnt[((size_t)ts * nseg + sg) * SCENE_INLINE_MAX];
      if (sg < seg) bef += c;
      tot += c;
    }
    running[0] = bef;
    if (seg == 0) pb.n_live[ts] = tot;
  }
  __syncthreads();
  int buf = 0;
  for (int base = lo; base < hi; base += CMP_T, buf ^= 1) {  // one barrier per 1024-slot chunk
    const int i = base + tid;
    const int id = i < hi ? qs[i] : -1;
    const unsigned b = __ballot_sync(0xffffffffu, id >= 0);
    if (lane == 0) wtot[buf][warp] = __popc(b);
    __syncthreads();
    int off = running[buf] + __popc(b & ((1u << lane) - 1));
    for (int w = 0; w < warp; ++w) off += wtot[buf][w];
    if (id >= 0) ql[off] = id;
    if (tid == CMP_T - 1) running[buf ^ 1] = off + (id >= 0 ? 1 : 0);  // last thread's end offset = new running total
  }
}

// ------------------------------------------------------------------------------------------
// K7 film resolve: Tile::add_sample (film.rs:167-172, :54-61) + copy_from_tile (:82-98).
// The reference adds a pixel's samples in wavefront order: by depth, then by shading-slot order inside
// the tile.  Each path recorded (depth, slot) when it terminated and its depth-0 slot, so ONE WARP per
// pixel orders the pixel's spp paths by those keys (in shared memory: 12 B per path; skipped when they
// already are in order) and 9 lanes run the 9 channel sums strictly sequentially in that order, gathering
// the payload from L2 -> bit-identical film, no float atomics, deterministic across runs, pass sizes and
// GPU counts.  Then / spp.  (Round 1 used one 128-thread CTA per pixel with <= 6 busy threads: 8-11 % of
// HBM; one warp per pixel puts 4-16x more pixels in flight per SM.)
// ------------------------------------------------------------------------------------------
#define RES_MAX_WARPS 8
#define RES_BINS 512  // histogram bins of the radix sort (digits of up to 9 bits)
#define RES_ROW 33                       // staging rows are 32 entries + 1 pad: the channel lanes read their rows bank-conflict free
#define RES_STAGE_FLOATS (6 * RES_ROW + 2)  // staging buffer of the ordered sums: up to 6 channel rows
// per warp: key[np] (by sample index), two index arrays (ping-pong of the radix sort), the histogram bins, the staging rows
__host__ __device__ inline size_t resolve_smem_per_warp(int np) {
  return (size_t)np * (sizeof(uint32_t) + 2 * sizeof(uint16_t)) + RES_BINS * sizeof(int) + RES_STAGE_FLOATS * sizeof(float);
}
static inline int resolve_warps_per_cta(int np) {
  int w = (int)((size_t)200 * 1024 / resolve_smem_per_warp(np));
  return w < 1 ? 0 : (w > RES_MAX_WARPS ? RES_MAX_WARPS : w);
}
// One warp sorts the n sample indices in src[] by key[index] ascending: LSD radix sort over the low key_bits bits, stable, in
// ceil(key_bits / 9) passes of equal digit width (<= 9 bits), passes whose digit is the same for every key are skipped.
// Returns the array that holds the result (src or tmp).  (The bitonic network it replaces needed 78 dependent shared-memory
// stages at 4096 spp - 400 k cycles per pixel at two warps per scheduler.)
RT_D uint16_t* warp_radix_sort(const uint32_t* key, uint16_t* src, uint16_t* tmp, int n, int key_bits, int lane, int* hist) {
  const unsigned lt = (1u << lane) - 1u;
  const int passes = (key_bits + 8) / 9, dbits = (key_bits + passes - 1) / passes;  // digit width <= 9
  const unsigned dmask = (1u << dbits) - 1u;
  const int per_lane = (1 << dbits) >> 5;  // bins owned by a lane in the scan (dbits >= 5 as long as key_bits >= 5)
  for (int shift = 0; shift < key_bits; shift += dbits) {
    for (int b = lane; b <= (int)dmask; b += 32) hist[b] = 0;
    __syncwarp();
#pragma unroll 4
    for (int base = 0; base < n; base += 32) {
      const int i = base + lane;
      if (i < n) atomicAdd(&hist[(key[src[i]] >> shift) & dmask], 1);
    }
    __syncwarp();
    // exclusive scan of the bins: lane l owns bins per_lane * l .. per_lane * (l + 1) - 1
    int sum = 0;
    bool uniform = false;
    for (int q = 0; q < per_lane; ++q) {
      const int c = hist[per_lane * lane + q];
      uniform |= c == n;
      sum += c;
    }
    if (__any_sync(0xffffffffu, uniform)) continue;  // every key has the same digit here: nothing to do
    int incl = sum;
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    int run = incl - sum;
    for (int q = 0; q < per_lane; ++q) {
      const int c = hist[per_lane * lane + q];
      hist[per_lane * lane + q] = run;
      run += c;
    }
    __syncwarp();
    for (int base = 0; base < n; base += 32) {
      const int i = base + lane;
      const bool act = i < n;
      const int v = act ? src[i] : 0;
      const unsigned d = act ? ((key[v] >> shift) & dmask) : (RES_BINS + lane);  // inactive lanes: singleton groups
      const unsigned m = __match_any_sync(0xffffffffu, d);
      const int leader = __ffs(m) - 1;
      int pos = 0;
      if (act && lane == leader) {
        pos = hist[d];
        hist[d] = pos + __popc(m);
      }
      pos = __shfl_sync(0xffffffffu, pos, leader) + __popc(m & lt);
      if (act) tmp[pos] = (uint16_t)v;
      __syncwarp();
    }
    uint16_t* t = src;
    src = tmp;
    tmp = t;
  }
  return src;
}
// keys of one order into shared memory (key[sample index]) and the indices of the samples that take part, in sample order,
// into idx[]; returns their number, *unordered != 0 if their keys are not ascending already.
// WHICH = 0: depth-0 slot + 1 of receives_light hits (WorldNormal / Alpha order, integrator.rs:161-169);
// WHICH = 1: (depth, slot) at termination (Color / Background order, integrator.rs:178-203), packed as depth << slot_bits | slot
// (slot < 2^slot_bits) so that the radix sort sees as few significant bits as possible.
template <int WHICH>
RT_D int resolve_keys(const float4* __restrict__ nrm0, const uint32_t* __restrict__ term, const float4* __restrict__ prefetch, int spp, int slot_bits,
                      int lane, uint32_t* key, uint16_t* idx, int* unordered) {
  const unsigned lt = (1u << lane) - 1u;
  int n = 0, bad = 0;
  uint32_t prev = 0;  // largest key so far (keys ascend as long as nothing is `bad`)
  for (int base = 0; base < spp; base += 32) {
    const int i = base + lane;
    uint32_t k = 0xffffffffu;
    if (i < spp) {
      if (WHICH == 0) {
        const uint32_t s0 = __float_as_uint(nrm0[i].w);
        if (s0) k = s0;
      } else {
        const uint32_t t = term[i];
        if (t >> 30) k = (((t >> TERM_DEPTH_SHIFT) & 0xffu) << slot_bits) | (t & (TERM_MAX_SLOTS - 1u));  // same order, fewer significant bits
        asm volatile("prefetch.global.L2 [%0];" ::"l"(prefetch + i));  // the payload the ordered sum will gather (same pixel, permuted order)
      }
      key[i] = k;
    }
    const bool valid = k != 0xffffffffu;
    const unsigned vm = __ballot_sync(0xffffffffu, valid);
    if (valid) idx[n + __popc(vm & lt)] = (uint16_t)i;
    // sortedness among the valid keys: compare with the previous valid key (of this chunk, else of earlier chunks)
    const unsigned below = vm & lt;
    const int pl = below ? 31 - __clz(below) : -1;
    const uint32_t pk_in = __shfl_sync(0xffffffffu, k, pl < 0 ? 0 : pl);
    const uint32_t pk = pl < 0 ? prev : pk_in;
    bad |= valid && (n + __popc(below) > 0) && pk > k;
    if (vm) prev = __shfl_sync(0xffffffffu, k, 31 - __clz(vm));
    n += __popc(vm);
  }
  *unordered = __any_sync(0xffffffffu, bad);
  return n;
}
// Strictly sequential float sums over the n entries of order[] (the reference's accumulation order), channel lanes
// [0, n_rows): row r of the staging buffer holds, for 32 entries at a time, the value lane r has to add - component r % 3 of
// src[order[i]] if the entry's class matches the row's (`want_lo` for rows 0-2, `want_hi` for rows 3-5; < 0: every entry), else
// +0.0f (an exact no-op: the accumulator can never be -0).  The payload is gathered by the whole warp (32 loads in flight, the
// next chunk already requested), so the sum itself is one dependent FADD chain per channel fed from shared memory.
RT_D float resolve_sum(const float4* __restrict__ src, const uint32_t* __restrict__ term, const uint16_t* order, int n, int lane, int n_rows,
                       int want_lo, int want_hi, float* stage) {
  auto fetch = [&](int base) {
    float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    const int i = base + lane;
    if (i < n) {
      const int p = order[i];
      v = src[p];
      v.w = term ? __uint_as_float(term[p] >> 30) : 0.0f;
    }
    return v;
  };
  float acc = 0.0f;
  float4 cur = fetch(0), nxt = fetch(32);
  for (int base = 0; base < n; base += 32) {
    const float4 nxt2 = fetch(base + 64);  // two chunks in flight ahead of the one being summed
    const int kind = (int)__float_as_uint(cur.w);
    const bool lo = want_lo < 0 || kind == want_lo, hi = want_hi < 0 || kind == want_hi;
    stage[0 * RES_ROW + lane] = lo ? cur.x : 0.0f;
    stage[1 * RES_ROW + lane] = lo ? cur.y : 0.0f;
    stage[2 * RES_ROW + lane] = lo ? cur.z : 0.0f;
    if (n_rows > 3) {
      stage[3 * RES_ROW + lane] = hi ? cur.x : 0.0f;
      stage[4 * RES_ROW + lane] = hi ? cur.y : 0.0f;
      stage[5 * RES_ROW + lane] = hi ? cur.z : 0.0f;
    }
    __syncwarp();
    const int m = min(32, n - base);
    if (lane < n_rows) {
      const float* row = stage + lane * RES_ROW;
#pragma unroll 8
      for (int j = 0; j < m; ++j) acc += row[j];
    }
    __syncwarp();
    cur = nxt;
    nxt = nxt2;
  }
  return acc;
}
__global__ void __launch_bounds__(RES_MAX_WARPS * 32) k_resolve(const DevFrame fr, const PassBufs pb, float* __restrict__ color,
                                                                 float* __restrict__ alpha, float* __restrict__ background,
                                                                 float* __restrict__ normal, const int np, const int wpc, const int slot_bits,
                                                                 const int depth_bits) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* mine = smem_raw + (size_t)warp * resolve_smem_per_warp(np);
  float* stage = reinterpret_cast<float*>(mine);
  int* hist = reinterpret_cast<int*>(stage + RES_STAGE_FLOATS);
  uint32_t* key = reinterpret_cast<uint32_t*>(hist + RES_BINS);
  uint16_t* idx0 = reinterpret_cast<uint16_t*>(key + np);
  uint16_t* idx1 = idx0 + np;
  const int ts = blockIdx.y, pl = blockIdx.x * wpc + warp;
  const TileGeom tg = tile_geom(fr, pb.tile_ids[ts]);
  if (pl >= tg.tw * tg.th) return;  // warp-uniform
  const int xl = pl / tg.th, yl = pl - xl * tg.th;
  const size_t pix = (size_t)(tg.x0 + xl) + (size_t)(tg.y0 + yl) * fr.W;
  const size_t g0 = (size_t)ts * pb.R + (size_t)pl * fr.spp;
  const float4* __restrict__ nrm0 = pb.nrm0 + g0;
  const float4* __restrict__ rad = pb.rad + g0;
  const uint32_t* __restrict__ term = pb.term + g0;
  const float div = (float)fr.spp;
  int unordered;
  // WorldNormal xyz (lanes 0-2) and Alpha in depth-0 slot order
  {
    const int nA = resolve_keys<0>(nrm0, term, nrm0, fr.spp, slot_bits, lane, key, idx0, &unordered);
    __syncwarp();
    const uint16_t* order = unordered ? warp_radix_sort(key, idx0, idx1, nA, slot_bits + 1, lane, hist) : idx0;
    __syncwarp();
    const float acc = resolve_sum(nrm0, nullptr, order, nA, lane, 3, -1, -1, stage);
    if (lane < 3 && normal) normal[3 * pix + lane] = acc / div;
    if (lane == 3 && alpha) alpha[pix] = (float)nA / div;  // Alpha(1.0) per depth-0 receives_light sample: a sum of nA ones is nA exactly
  }
  __syncwarp();
  // Color rgb (lanes 0-2) and Background rgb (lanes 3-5) in (depth, slot) order
  {
    const int nB = resolve_keys<1>(nrm0, term, rad, fr.spp, slot_bits, lane, key, idx0, &unordered);
    __syncwarp();
    const uint16_t* order = unordered ? warp_radix_sort(key, idx0, idx1, nB, slot_bits + depth_bits, lane, hist) : idx0;
    __syncwarp();
    const float acc = resolve_sum(rad, term, order, nB, lane, 6, (int)TERM_COLOR, (int)TERM_BACKGROUND, stage);
    float* dst = lane < 3 ? color : background;
    if (lane < 6 && dst) dst[3 * pix + lane % 3] = acc / div;
  }
}

// ------------------------------------------------------------------------------------------
// multi-GPU film gather helpers.  Slab layout [k][10][tile_w*tile_h], k = rank-local tile ordinal, pixel order
// x + y*tile_w, channel order color rgb, alpha, background rgb, normal xyz.  `tile_table` holds, for every rank r,
// `per_rank` entries (its ascending tile indices, padded with -1); slab of rank r starts at r * per_rank * 10 * tp.
// pack: this rank's tiles -> its slab (grid.x = per_rank, rank = first_rank).  unpack: ONE launch over all ranks'
// slabs (grid.x = world * per_rank), skipping `skip_rank` (the local one, already in the planes).
// Tiles are disjoint (film.rs:82-98): the gather moves bytes, it never reduces.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_film_slab(int W, int H, int tile_w, int tile_h, int nty, const int* __restrict__ tile_table, int per_rank,
                                                   int first_rank, int skip_rank, int unpack, float* __restrict__ slabs, float* color, float* alpha,
                                                   float* background, float* normal) {
  const int b = blockIdx.x + first_rank * per_rank;
  if (b / per_rank == skip_rank) return;
  const int tile_id = tile_table[b];
  if (tile_id < 0) return;
  const int tx = tile_id / nty, ty = tile_id % nty;
  const int x0 = tx * tile_w, y0 = ty * tile_h;
  const int tp = tile_w * tile_h;
  float* sl = slabs + (size_t)b * 10 * tp;
  for (int p = threadIdx.x; p < tp; p += blockDim.x) {
    const int xl = p % tile_w, yl = p / tile_w;
    const int x = x0 + xl, y = y0 + yl;
    if (x >= W || y >= H) {
      if (!unpack)
        for (int c = 0; c < 10; ++c) sl[c * tp + p] = 0.0f;
      continue;
    }
    const size_t pix = (size_t)x + (size_t)y * W;
    if (!unpack) {
      for (int c = 0; c < 3; ++c) sl[c * tp + p] = color ? color[3 * pix + c] : 0.0f;
      sl[3 * tp + p] = alpha ? alpha[pix] : 0.0f;
      for (int c = 0; c < 3; ++c) sl[(4 + c) * tp + p] = background ? background[3 * pix + c] : 0.0f;
      for (int c = 0; c < 3; ++c) sl[(7 + c) * tp + p] = normal ? normal[3 * pix + c] : 0.0f;
    } else {
      if (color) for (int c = 0; c < 3; ++c) color[3 * pix + c] = sl[c * tp + p];
      if (alpha) alpha[pix] = sl[3 * tp + p];
      if (background) for (int c = 0; c < 3; ++c) background[3 * pix + c] = sl[(4 + c) * tp + p];
      if (normal) for (int c = 0; c < 3; ++c) normal[3 * pix + c] = sl[(7 + c) * tp + p];
    }
  }
}
// pixels outside the reference's tile grid (film.rs:399-404 drops the last partial tile when 0 < res % tile < tile/2) are
// never written by a render; device-space planes are cleared there so they do not keep stale caller data (host-space
// planes start from zeros anyway).
__global__ void __launch_bounds__(256) k_zero_uncovered(int W, int H, int cov_w, int cov_h, float* color, float* alpha, float* background, float* normal) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)W * H) return;
  const int x = (int)(i % W), y = (int)(i / W);
  if (x < cov_w && y < cov_h) return;
  if (alpha) alpha[i] = 0.0f;
  for (int c = 0; c < 3; ++c) {
    if (color) color[3 * i + c] = 0.0f;
    if (background) background[3 * i + c] = 0.0f;
    if (normal) normal[3 * i + c] = 0.0f;
  }
}

// ------------------------------------------------------------------------------------------
// Film post-process (SURVEY §8f rank 3): the per-pixel arithmetic of Film::save_to, film.rs:205-377.
// One thread per output pixel; a streaming kernel (<= 28 B in, <= 4 B out per pixel).
// ------------------------------------------------------------------------------------------
// f32 scalar semantics of the reference: `x.max(0.0).min(1.0)` and `(v*255.0).min(255.0).max(0.0) as u8`
// use Rust's f32::min/max (NaN loses) and a saturating, truncating cast.
__host__ __device__ inline float post_saturate(float x) {
  float a = (x != x) ? 0.0f : (x > 0.0f ? x : 0.0f);
  return a < 1.0f ? a : 1.0f;
}
__host__ __device__ inline float post_gamma(float x) { return dm::pow(x, 1.0f / 2.2f); }  // spectrum.rs:30-32
__host__ __device__ inline unsigned char post_u8(float v) {
  float a = v * 255.0f;
  a = (a != a) ? 255.0f : (a < 255.0f ? a : 255.0f);
  a = a > 0.0f ? a : 0.0f;
  return (unsigned char)(int)a;
}
__host__ __device__ inline int post_bytes_per_pixel(int mode) { return mode == RAYN_POST_COLOR_ALPHA ? 4 : (mode == RAYN_POST_ALPHA ? 1 : 3); }
__host__ __device__ inline void post_pixel(int mode, const float* __restrict__ color, const float* __restrict__ alpha,
                                           const float* __restrict__ background, const float* __restrict__ normal, size_t src,
                                           unsigned char* dst) {
  switch (mode) {
    case RAYN_POST_COLOR_PLUS_BACKGROUND:
      for (int c = 0; c < 3; ++c) dst[c] = post_u8(post_gamma(post_saturate(color[3 * src + c] + background[3 * src + c])));
      break;
    case RAYN_POST_COLOR_ALPHA:
      for (int c = 0; c < 3; ++c) dst[c] = post_u8(post_gamma(post_saturate(color[3 * src + c])));
      dst[3] = post_u8(alpha[src]);
      break;
    case RAYN_POST_COLOR_ONLY:
      for (int c = 0; c < 3; ++c) dst[c] = post_u8(post_gamma(color[3 * src + c]));
      break;
    case RAYN_POST_BACKGROUND:
      for (int c = 0; c < 3; ++c) dst[c] = post_u8(post_gamma(post_saturate(background[3 * src + c])));
      break;
    case RAYN_POST_WORLD_NORMAL:
      for (int c = 0; c < 3; ++c) dst[c] = post_u8(normal[3 * src + c] * 0.5f + 0.5f);
      break;
    default:
      dst[0] = post_u8(alpha[src]);
  }
}
__global__ void __launch_bounds__(256) k_postprocess(int mode, int W, int H, const float* __restrict__ color, const float* __restrict__ alpha,
                                                     const float* __restrict__ background, const float* __restrict__ normal,
                                                     unsigned char* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)W * H) return;
  const int x = (int)(i % W), y = (int)(i / W);
  const size_t src = (size_t)x + (size_t)(H - 1 - y) * W;  // film.rs:236
  unsigned char px[4];
  post_pixel(mode, color, alpha, background, normal, src, px);
  const int bpp = post_bytes_per_pixel(mode);
  for (int c = 0; c < bpp; ++c) out[(size_t)i * bpp + c] = px[c];
}

// ------------------------------------------------------------------------------------------
// Device-side sampler state (SURVEY §8f rank 2): the same R_d tables and SmallRng scramble as
// host_inputs.cpp, generated in HBM so an 8K frame does not upload a 133 MB scramble plane.
// Integer arithmetic only -> bit-identical to the host builders (tests compare them).
// ------------------------------------------------------------------------------------------
RT_D float dev_rd_value(unsigned long long alpha, unsigned long long n) {
  const unsigned long long frac = alpha * n + 0x8000000000000000ull;
  return (float)(frac >> 40) * (1.0f / 16777216.0f);
}
__global__ void __launch_bounds__(256) k_gen_rd_tables(int spp, int sets_1d, int sets_2d, unsigned long long offset, float* __restrict__ s1,
                                                       float* __restrict__ s2) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long n1 = (long long)spp * sets_1d, n2 = (long long)spp * sets_2d;
  if (i < n1) {
    const int set = (int)(i / spp), n = (int)(i % spp);
    s1[i] = dev_rd_value(0x9e3779b97f4a7c15ull, ((offset + (unsigned long long)set) << 32) + (unsigned long long)n + 1ull);
  } else if (i < n1 + n2) {
    const long long j = i - n1;
    const int set = (int)(j / spp), n = (int)(j % spp);
    const unsigned long long base = ((offset + (unsigned long long)sets_1d + (unsigned long long)set) << 32) + (unsigned long long)n + 1ull;
    s2[2 * j + 0] = dev_rd_value(0xc13fa9a902a6328full, base);
    s2[2 * j + 1] = dev_rd_value(0x91e10da5c79e7b1cull, base);
  }
}
__global__ void __launch_bounds__(256) k_gen_scramble(int W, int H, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)W * H) return;
  // rand_core 0.5.1 seed_from_u64 (PCG32 expansion) -> rand_pcg 0.2.1 Mcg128Xsl64 -> first f32 (film.rs:460-461)
  unsigned long long state = (unsigned long long)i;  // x + y*width
  unsigned int sd[4];
  for (int c = 0; c < 4; ++c) {
    state = state * 6364136223846793005ull + 11634580027462260723ull;
    const unsigned int xorshifted = (unsigned int)(((state >> 18) ^ state) >> 27);
    const unsigned int rot = (unsigned int)(state >> 59);
    sd[c] = (xorshifted >> rot) | (xorshifted << ((32 - rot) & 31));
  }
  unsigned __int128 s = ((unsigned __int128)(((unsigned long long)sd[3] << 32) | sd[2]) << 64) | (((unsigned long long)sd[1] << 32) | sd[0]);
  s |= 1;
  s = s * (((unsigned __int128)2549297995355413924ull << 64) | 4865540595714422341ull);
  const unsigned int r2 = (unsigned int)(s >> 122);
  const unsigned long long xsl = (unsigned long long)(s >> 64) ^ (unsigned long long)s;
  const unsigned long long o = (xsl >> r2) | (xsl << ((64 - r2) & 63));
  out[i] = (float)(((unsigned int)o) >> 8) * (1.0f / 16777216.0f);
}

// ------------------------------------------------------------------------------------------
// known-answer kernels (tests only)
// ------------------------------------------------------------------------------------------
__global__ void k_kat_detmath(int op, long long n, const float* a, const float* b, float* out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s, c;
  switch (op) {
    case 0: out[i] = dm::exp(a[i]); break;
    case 1: out[i] = dm::ln(a[i]); break;
    case 2: out[i] = dm::pow(a[i], b[i]); break;
    case 3: dm::sincos(a[i], &s, &c); out[i] = s; break;
    case 4: dm::sincos(a[i], &s, &c); out[i] = c; break;
    case 5: out[i] = dm::tan(a[i]); break;
    case 6: out[i] = dm::atan2(a[i], b[i]); break;
    case 7: out[i] = dm::powi5(a[i]); break;
  }
}
__global__ void k_kat_sdf_dist(const RaynHitable h, long long n, const float* p3, float* out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = sdf_dist(h, mk3(p3[3 * i], p3[3 * i + 1], p3[3 * i + 2]));
}
// packed estimator of the march kernels vs the scalar one: out = sdf_dist2<V>(p[2i], p[2i+1]) per pair; n even
template <int V>
__global__ void k_kat_sdf_dist2(const RaynHitable h, const float one, long long n, const float* p3, float* out) {
  const long long i = 2 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= n) return;
  const SdfK k = make_sdfk(h, one);
  const long long j = i + 1 < n ? i + 1 : i;
  int it = 0;
  const float2 d = sdf_dist2<V>(k, f2(p3[3 * i], p3[3 * j]), f2(p3[3 * i + 1], p3[3 * j + 1]), f2(p3[3 * i + 2], p3[3 * j + 2]), it);
  out[i] = d.x;
  if (i + 1 < n) out[i + 1] = d.y;
}
// Newton division of rt_sdf2.cuh vs IEEE division: counts mismatches of num / x over the n consecutive floats starting at bit pattern first_bits
__global__ void k_kat_fastdiv(float num, unsigned first_bits, long long n, unsigned long long* mismatches) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  int bad = 0;
  if (i < n) {
    const float x = __uint_as_float(first_bits + (unsigned)i);
    const float2 q = fastdiv2(num, f2(x, x));
    const float ref = num / x;
    bad = (__float_as_uint(q.x) != __float_as_uint(ref)) + (__float_as_uint(q.y) != __float_as_uint(ref)) +
          (__float_as_uint(fastdiv1(num, x)) != __float_as_uint(ref));
  }
  warp_add(mismatches, bad);
}
// rt_sdf2.cuh::fastdiv2_3 against IEEE division over n consecutive divisors (grid-stride): the check behind the DIV3 variants
__global__ void __launch_bounds__(256) k_verify_div3(float num, unsigned first_bits, unsigned long long n, unsigned long long* mismatches) {
  int bad = 0;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
    const float x = __uint_as_float(first_bits + (unsigned)i);
    const float2 q = fastdiv2_3(num, f2(x, x));
    const float ref = num / x;
    bad += (__float_as_uint(q.x) != __float_as_uint(ref)) | (__float_as_uint(q.y) != __float_as_uint(ref)) |
           (__float_as_uint(fastdiv1_3(num, x)) != __float_as_uint(ref));
  }
  warp_add(mismatches, bad);
}
__global__ void k_kat_sdf_hit(const RaynHitable h, const RaynRenderConsts rc, long long n, const float* o3, const float* d3,
                              const float* t_max, Thr thr, float* out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int ev = 0;
  out[i] = sdf_hit(h, rc, mk3(o3[3 * i], o3[3 * i + 1], o3[3 * i + 2]), mk3(d3[3 * i], d3[3 * i + 1], d3[3 * i + 2]), t_max[i],
                   thr, &ev);
}
template <class Scn>
__global__ void k_kat_occluded(const __grid_constant__ Scn sc, long long n, const float* s3, const float* e3, float* out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int ev = 0;
  // reference semantics: product over all hitables (no reordering) - used to validate the
  // early-out form in test_occluded as well
  float acc = 1.0f;
  const f3 a = mk3(s3[3 * i], s3[3 * i + 1], s3[3 * i + 2]), b = mk3(e3[3 * i], e3[3 * i + 1], e3[3 * i + 2]);
  for (int k = 0; k < sc.n_hit; ++k)
    acc = acc * (sc.hit[k].kind == RAYN_HITABLE_SPHERE ? sphere_occluded(sc.hit[k], a, b, 0.0f) : sdf_occluded(sc.hit[k], sc.rc, a, b, &ev));
  const float fast = test_occluded(sc, a, b, &ev);
  out[i] = acc == fast ? acc : -1.0f;  // -1 flags a disagreement between the two forms
}
template __global__ void k_kat_occluded<DevScene>(const __grid_constant__ DevScene, long long, const float*, const float*, float*);
template <class Scn>
__global__ void k_kat_closest_hit(const __grid_constant__ Scn sc, Thr thr, long long n, const float* o3, const float* d3,
                                  float* out_t, int* out_obj) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int ev = 0;
  closest_hit(sc, mk3(o3[3 * i], o3[3 * i + 1], o3[3 * i + 2]), mk3(d3[3 * i], d3[3 * i + 1], d3[3 * i + 2]), thr, &out_t[i],
              &out_obj[i], &ev);
}
template __global__ void k_kat_closest_hit<DevScene>(const __grid_constant__ DevScene, Thr, long long, const float*, const float*, float*, int*);

__global__ void k_kat_light_sample(const RaynLight L, long long n, const float* s0, const float* s1, const float* p3, float* out_pt3, float* out_pdf) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  f3 pt, li;
  float pdf;
  light_sample(L, s0[i], s1[i], mk3(p3[3 * i], p3[3 * i + 1], p3[3 * i + 2]), &pt, &li, &pdf);
  out_pt3[3 * i] = pt.x, out_pt3[3 * i + 1] = pt.y, out_pt3[3 * i + 2] = pt.z;
  out_pdf[i] = pdf;
}
__global__ void k_kat_light_sample_volume(const RaynLight L, long long n, const float* sample, const float* o3, const float* d3, const float* t_max,
                                          float* out_t, float* out_pdf) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  light_sample_volume(L, sample[i], mk3(o3[3 * i], o3[3 * i + 1], o3[3 * i + 2]), mk3(d3[3 * i], d3[3 * i + 1], d3[3 * i + 2]), t_max[i], &out_t[i],
                      &out_pdf[i]);
}
__global__ void k_kat_bsdf(const RaynMaterial m, long long n, const float* n3, const float* wo3, const float* s1d, const float* u4, float* out_wi3,
                           float* out_f3, float* out_pdf, float* out_fe3) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ShadingPoint sp;
  sp.normal = mk3(n3[3 * i], n3[3 * i + 1], n3[3 * i + 2]);
  sp.basis = onb(sp.normal);
  const f3 wo = mk3(wo3[3 * i], wo3[3 * i + 1], wo3[3 * i + 2]);
  const Scatter se = bsdf_scatter(m, wo, sp, s1d[i], u4[4 * i], u4[4 * i + 1], u4[4 * i + 2], u4[4 * i + 3]);
  const f3 fe = bsdf_f(m, wo, se.wi, sp.normal);
  out_wi3[3 * i] = se.wi.x, out_wi3[3 * i + 1] = se.wi.y, out_wi3[3 * i + 2] = se.wi.z;
  out_f3[3 * i] = se.f.x, out_f3[3 * i + 1] = se.f.y, out_f3[3 * i + 2] = se.f.z;
  out_fe3[3 * i] = fe.x, out_fe3[3 * i + 1] = fe.y, out_fe3[3 * i + 2] = fe.z;
  out_pdf[i] = se.pdf;
}

}  // namespace rt

