// api.cu — C-ABI implementation (include/rayn_b200.h): context, scene upload, the tile-pass
// scheduler that drives the wavefront kernels, the NCCL film gather and the known-answer
// entry points.  No torch types, no exceptions across the boundary.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <limits.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <vector>

#include "rt_kernels.cuh"
#ifdef RAYN_LEGACY_KERNELS
#include "rt_legacy.cuh"
#endif

using namespace rt;

static thread_local std::string g_last_error;

struct TimedLaunch {
  int kernel;
  cudaEvent_t a, b;
};

// ---- NCCL, resolved at run time (no link-time dependency: the library must load on a box without NCCL) ----
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[RAYN_COMM_ID_BYTES]; } ncclUniqueId;
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static const int kNcclFloat = 7;  // ncclFloat32

struct RaynComm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 0;
  // shard tables of the last geometry gathered
  int W = 0, H = 0, tw = 0, th = 0, per_rank = 0;
  std::vector<std::vector<int>> shards;
  int* d_table = nullptr;   // [world * per_rank], -1 padded
  float* d_slabs = nullptr; // [world * per_rank * 10 * tw * th]
  size_t cap_slabs = 0;
};

struct RaynContext {
  int device = 0;
  int flags = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  bool has_scene = false;
  DevScene scene;  // every field of the uploaded scene; the arrays only when it takes the inline path (!tables)
  // large-scene path (more than SCENE_INLINE_MAX hitables, materials or lights, or RAYN_FLAG_SCENE_TABLES): the kernels take
  // tscene, whose tables live in d_tables.  scene_gen counts uploads, so that a graph captured for other table contents
  // is never replayed (the tables are rewritten in place; their pointers do not change).
  bool tables = false;
  TableScene tscene;
  unsigned char* d_tables = nullptr;
  size_t cap_tables = 0;
  uint64_t scene_gen = 0;
  std::vector<RaynHitable> h_hit;  // host copies of the uploaded descriptors (launch decisions)
  std::vector<RaynMaterial> h_mat;
  int64_t cap_paths = 0;  // requested paths per pass
  // pass buffers
  int64_t alloc_paths = 0, alloc_q = 0, alloc_seg = 0;
  int alloc_lc_ns = 0;
  int alloc_tiles = 0;
  int64_t alloc_segcnt = 0;  // ints in PassBufs::seg_cnt
  int64_t alloc_bins = 0;    // ints in PassBufs::bin_start
  size_t pass_bytes = 0;
  PassBufs pb;
  int* d_tile_ids = nullptr;
  int* d_batch_prefix = nullptr;  // [alloc_tiles + 1]
  int* d_work_ctr = nullptr;      // [WC_TOTAL] global work counters of the persistent kernels
  int n_sm = 148;
  struct Occ {  // resident CTAs per SM of the persistent and work-list kernels, per scene type ([0] DevScene, [1] TableScene)
    int ext[SDFV_COUNT], shd[SDFV_COUNT], nrm[SDFV_COUNT];
    int pre = 8, post = 8, sph = 8;
  } occ[2];
  int sdf_var[RAYN_MAX_HITABLES];  // march-kernel variant of every SDF hitable of the uploaded scene (rt_sdf2.cuh::sdf_variant)
  struct Div3Check { float min_r2, fixed_r2; bool ok; };
  std::vector<Div3Check> div3_cache;  // exhaustive fastdiv2_3 checks already run on this device
  // staging for host-space inputs / outputs
  float *d_s1 = nullptr, *d_s2 = nullptr, *d_scr = nullptr, *d_fis = nullptr;
  size_t cap_s1 = 0, cap_s2 = 0, cap_scr = 0;
  float* d_planes = nullptr;
  size_t cap_planes = 0;
  int* d_pack_ids = nullptr;
  size_t cap_pack_ids = 0;
  unsigned char* d_post = nullptr;
  size_t cap_post = 0;
  unsigned long long* d_kat = nullptr;
  RaynStats stats;
  bool qlog_enabled = false;
  std::vector<int32_t> qlog;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<TimedLaunch> timed;
  size_t timed_used = 0;
  // a render that has been enqueued but not finished
  bool pending = false;
  std::vector<int> job_tiles;
  int job_w = 0, job_h = 0, job_tw = 0, job_th = 0, job_spp = 0, job_nty = 0;
  unsigned long long h_counters[CNT_TOTAL];
  RaynComm comm;
  // CUDA graph of the last small single-pass frame (launch-bound frames: the whole per-depth kernel sequence replays as one launch)
  cudaGraphExec_t graph_exec = nullptr;
  uint64_t graph_key = 0;
  RaynStats graph_stats;  // launch counts recorded while capturing
};

static uint64_t fnv1a(uint64_t h, const void* data, size_t n) {
  const unsigned char* p = (const unsigned char*)data;
  for (size_t i = 0; i < n; ++i) h = (h ^ p[i]) * 1099511628211ull;
  return h;
}

static int32_t fail(RaynContext* ctx, int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
  if (ctx) ctx->err = buf;
  return code;
}
// a failing runtime call leaves a sticky per-thread "last error": clear it when reporting, or the next valid call's
// cudaGetLastError() check would fail spuriously
#define CU(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) {                                                                         \
      cudaGetLastError();                                                                            \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? RAYN_ERR_OOM : RAYN_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                  cudaGetErrorString(e_), __FILE__, __LINE__);                                       \
    }                                                                                                \
  } while (0)
#define NC(call)                                                                                     \
  do {                                                                                               \
    int r_ = (call);                                                                                 \
    if (r_ != 0)                                                                                     \
      return fail(ctx, RAYN_ERR_NCCL, "%s: %s (%s:%d)", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?", __FILE__, __LINE__); \
  } while (0)

template <class T>
static cudaError_t regrow(T** p, size_t* cap, size_t need) {
  if (need <= *cap && *p) return cudaSuccess;
  if (*p) cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(need, 1) * sizeof(T));
  if (e == cudaSuccess) *cap = need;
  return e;
}

static void free_pass(RaynContext* c) {
  PassBufs& p = c->pb;
  cudaFree(p.o_time), cudaFree(p.d_t), cudaFree(p.rad), cudaFree(p.thr), cudaFree(p.nrm0), cudaFree(p.term);
  cudaFree(p.q_live), cudaFree(p.q_key), cudaFree(p.q_shade), cudaFree(p.n_live), cudaFree(p.n_slots), cudaFree(p.bin_start);
  cudaFree(c->d_tile_ids);
  cudaFree(c->d_batch_prefix);
  c->d_batch_prefix = nullptr;
  cudaFree(p.nrm), cudaFree(p.vis), cudaFree(p.seg_a), cudaFree(p.seg_b), cudaFree(p.lc_c), cudaFree(p.lc_t), cudaFree(p.seg_cnt), cudaFree(p.slot_prefix);
  unsigned long long* counters = p.counters;
  memset(&p, 0, sizeof p);
  p.counters = counters;
  c->d_tile_ids = nullptr;
  c->alloc_paths = c->alloc_q = c->alloc_seg = 0;
  c->alloc_lc_ns = 0;
  c->alloc_tiles = 0;
  c->alloc_segcnt = 0;
  c->alloc_bins = 0;
  c->pass_bytes = 0;
}

// bytes of pass state per path (what ensure_pass allocates), used to size passes against free device memory; the per-tile
// tables (bin starts and segment counts, maxk + 1 and maxk ints per row) are spread over the tile's R paths
static size_t pass_bytes_per_path(int R, int QS, int seg_per_path, int lc_ns, int maxk) {
  const double tile_ints = (double)(maxk + 1) + (double)((QS + SEG_SLOTS - 1) / SEG_SLOTS) * maxk;
  return 6 * sizeof(float4) + 2 * sizeof(uint32_t) + 2 * sizeof(int) + (size_t)(((double)QS / R) * sizeof(int) + 1) + (size_t)lc_ns * sizeof(float4) +
         (lc_ns > 4 ? 8 * sizeof(float) : 0) + (size_t)seg_per_path * 2 * sizeof(float4) + (size_t)(tile_ints * sizeof(int) / R + 1);
}

static int32_t ensure_pass(RaynContext* ctx, int n_tiles, int R, int QS, int seg_per_path_total, int n_sdf, int lc_ns, int maxk) {
  const int64_t need_paths = (int64_t)n_tiles * R, need_q = (int64_t)n_tiles * QS;
  const int64_t need_seg = need_paths * seg_per_path_total;  // all SDF queues together
  const int64_t need_segcnt = (int64_t)n_tiles * ((QS + SEG_SLOTS - 1) / SEG_SLOTS) * maxk;
  const int64_t need_bins = (int64_t)n_tiles * (maxk + 1);
  if (need_paths <= ctx->alloc_paths && need_q <= ctx->alloc_q && n_tiles <= ctx->alloc_tiles && need_seg <= ctx->alloc_seg && lc_ns <= ctx->alloc_lc_ns &&
      need_segcnt <= ctx->alloc_segcnt && need_bins <= ctx->alloc_bins)
    return RAYN_OK;
  free_pass(ctx);
  PassBufs& p = ctx->pb;
  size_t total = 0;
#define PASS_ALLOC(ptr, bytes)                                    \
  do {                                                            \
    cudaError_t e_ = cudaMalloc((void**)&(ptr), (size_t)(bytes)); \
    if (e_ != cudaSuccess) {                                      \
      cudaGetLastError();                                         \
      free_pass(ctx);                                             \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? RAYN_ERR_OOM : RAYN_ERR_CUDA, "pass buffers (%lld paths): %s", (long long)need_paths, cudaGetErrorString(e_)); \
    }                                                             \
    total += (size_t)(bytes);                                     \
  } while (0)
  PASS_ALLOC(p.o_time, need_paths * sizeof(float4));
  PASS_ALLOC(p.d_t, need_paths * sizeof(float4));
  PASS_ALLOC(p.rad, need_paths * sizeof(float4));
  PASS_ALLOC(p.thr, need_paths * sizeof(float4));
  PASS_ALLOC(p.nrm0, need_paths * sizeof(float4));
  PASS_ALLOC(p.term, need_paths * sizeof(uint32_t));
  PASS_ALLOC(p.q_live, need_paths * sizeof(int));
  PASS_ALLOC(p.q_key, need_paths * sizeof(int));
  PASS_ALLOC(p.q_shade, need_q * sizeof(int));
  PASS_ALLOC(p.n_live, n_tiles * sizeof(int));
  PASS_ALLOC(p.n_slots, n_tiles * sizeof(int));
  PASS_ALLOC(p.bin_start, (size_t)need_bins * sizeof(int));
  ctx->alloc_bins = need_bins;
  PASS_ALLOC(ctx->d_tile_ids, n_tiles * sizeof(int));
  PASS_ALLOC(ctx->d_batch_prefix, ((size_t)n_tiles + 1) * sizeof(int));
  PASS_ALLOC(p.seg_cnt, need_segcnt * sizeof(int));
  PASS_ALLOC(p.slot_prefix, (size_t)(1 + RAYN_MAX_SDF_HITABLES) * ((size_t)n_tiles + 1) * sizeof(int));
  p.prefix_stride = n_tiles + 1;
  ctx->alloc_segcnt = need_segcnt;
  PASS_ALLOC(p.nrm, need_paths * sizeof(float4));
  PASS_ALLOC(p.vis, need_paths * sizeof(uint32_t));
  if (need_seg > 0) {
    PASS_ALLOC(p.seg_a, need_seg * sizeof(float4));
    PASS_ALLOC(p.seg_b, need_seg * sizeof(float4));
  }
  p.seg_cap = n_sdf > 0 ? need_seg / n_sdf : 0;
  ctx->alloc_seg = need_seg;
  if (lc_ns > 0) {
    PASS_ALLOC(p.lc_c, need_paths * lc_ns * sizeof(float4));
    if (lc_ns > 4) PASS_ALLOC(p.lc_t, need_paths * 8 * sizeof(float));
  }
#undef PASS_ALLOC
  ctx->alloc_lc_ns = lc_ns;
  ctx->alloc_paths = need_paths;
  ctx->alloc_q = need_q;
  ctx->alloc_tiles = n_tiles;
  ctx->pass_bytes = total;
  return RAYN_OK;
}

static void timed_begin(RaynContext* ctx, int kernel) {
  if (!(ctx->flags & RAYN_FLAG_TIMING)) return;
  if (ctx->timed_used == ctx->timed.size()) {
    TimedLaunch t;
    t.kernel = kernel;
    cudaEventCreate(&t.a);
    cudaEventCreate(&t.b);
    ctx->timed.push_back(t);
  }
  ctx->timed[ctx->timed_used].kernel = kernel;
  cudaEventRecord(ctx->timed[ctx->timed_used].a, ctx->stream);
}
static void timed_end(RaynContext* ctx, int kernel, int launches = 1) {
  ctx->stats.launches += launches;
  ctx->stats.kernel_launches[kernel] += launches;
  if (!(ctx->flags & RAYN_FLAG_TIMING)) return;
  cudaEventRecord(ctx->timed[ctx->timed_used].b, ctx->stream);
  ctx->timed_used++;
}

struct DevTmp {
  std::vector<void*> ptrs;
  ~DevTmp() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <class T>
  T* up(const T* h, size_t n, cudaError_t* e) {
    T* d = nullptr;
    if (*e != cudaSuccess) return nullptr;
    *e = cudaMalloc((void**)&d, std::max<size_t>(n, 1) * sizeof(T));
    if (*e != cudaSuccess) return nullptr;
    ptrs.push_back(d);
    if (h) *e = cudaMemcpy(d, h, n * sizeof(T), cudaMemcpyHostToDevice);
    // cudaMemcpy from PAGEABLE memory returns once the data is staged; the DMA may still be in flight, and the test kernels
    // run on a non-blocking stream that does not order against the legacy stream: wait for the copy to land.
    if (h && *e == cudaSuccess) *e = cudaDeviceSynchronize();
    return d;
  }
};

// kernel launches specialised on the SDF variant (rt_sdf2.cuh)
#define DISPATCH_SDFV(v, STMT)                                                        \
  switch (v) {                                                                        \
    case SDFV_BOX_12_FAST: { constexpr int V = SDFV_BOX_12_FAST; STMT; } break;       \
    case SDFV_BOX_N_FAST: { constexpr int V = SDFV_BOX_N_FAST; STMT; } break;         \
    case SDFV_BULB: { constexpr int V = SDFV_BULB; STMT; } break;                     \
    case SDFV_BOX_12_DIV3: { constexpr int V = SDFV_BOX_12_DIV3; STMT; } break;       \
    case SDFV_BOX_N_DIV3: { constexpr int V = SDFV_BOX_N_DIV3; STMT; } break;         \
    default: { constexpr int V = SDFV_BOX_GENERIC; STMT; } break;                     \
  }

template <class S>
static cudaError_t query_occupancy(RaynContext::Occ& o) {
  cudaError_t e = cudaSuccess;
  for (int v = 0; v < SDFV_COUNT && e == cudaSuccess; ++v) {
    DISPATCH_SDFV(v, e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.ext[v], k_extend_march<V, S>, EXT_T, 0);
                  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.shd[v], k_shadow<V, S>, SHD_T, 0);
                  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.nrm[v], k_normals<V, S>, SLOT_BLOCK, 0));
  }
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.pre, k_shade_pre<S>, SLOT_BLOCK, 0);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.post, k_shade_post<S>, SLOT_BLOCK, 0);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.sph, k_extend_spheres<S>, EXT_BATCH, 0);
  return e;
}

static void tile_grid_of(int W, int H, int tw, int th, int* ntx, int* nty) {
  *ntx = (W + W % tw) / tw;  // film.rs:399-404
  *nty = (H + H % th) / th;
}
static std::vector<int> shard_of(int W, int H, int tw, int th, int rank, int world) {
  int ntx, nty;
  tile_grid_of(W, H, tw, th, &ntx, &nty);
  std::vector<int> v;
  for (int tx = 0; tx < ntx; ++tx)
    for (int ty = 0; ty < nty; ++ty)
      if ((tx + ty) % world == rank) v.push_back(tx * nty + ty);  // ascending: tile index = tx * nty + ty (film.rs:401-425)
  return v;
}

static int32_t render_enqueue(RaynContext* ctx, const RaynFrameDesc* f, const RaynFilmPlanes* out, const std::vector<int>* tiles_override,
                              RaynFilmPlanes* dev_planes_out);
static int32_t render_finish(RaynContext* ctx);
static int32_t gather_enqueue(RaynContext* ctx, int W, int H, int tw, int th, const RaynFilmPlanes* pl, bool in_group);

extern "C" {

int32_t rayn_b200_abi_version(void) { return RAYN_B200_ABI_VERSION; }
int32_t rayn_b200_muladd_fused(void) { return RAYN_MULADD_FUSED; }

const char* rayn_b200_last_error(const RaynContext* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

int32_t rayn_b200_create(const RaynConfig* cfg, RaynContext** out_ctx) {
  RaynContext* ctx = nullptr;
  if (!out_ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "out_ctx is NULL");
  *out_ctx = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, RAYN_ERR_NO_DEVICE, "no CUDA device: the rayn_b200 render path has no CPU fallback");
  }
  const int dev = cfg ? cfg->device : 0;
  if (dev < 0 || dev >= ndev) return fail(nullptr, RAYN_ERR_INVALID_ARG, "device %d out of range (have %d)", dev, ndev);
#ifndef RAYN_LEGACY_KERNELS
  if (cfg && (cfg->flags & RAYN_FLAG_SIMPLE_MARCH))
    return fail(nullptr, RAYN_ERR_UNSUPPORTED, "RAYN_FLAG_SIMPLE_MARCH needs the test build (librayn_b200_legacy.so, -DRAYN_LEGACY_KERNELS)");
#endif
  CU(cudaSetDevice(dev));
  ctx = new RaynContext();
  ctx->device = dev;
  ctx->flags = cfg ? cfg->flags : 0;
  ctx->cap_paths = (cfg && cfg->max_paths_per_pass > 0) ? cfg->max_paths_per_pass : (int64_t)96 << 20;  // fewer passes = fewer kernel tails (measured +3.5 %); clamped to free memory per frame
  memset(&ctx->pb, 0, sizeof ctx->pb);
  memset(&ctx->stats, 0, sizeof ctx->stats);
  memset(&ctx->scene, 0, sizeof ctx->scene);
  cudaError_t e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc(&ctx->pb.counters, CNT_TOTAL * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_fis, RAYN_FIS_TABLE_SIZE * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_work_ctr, WC_TOTAL * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_kat, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev1);
  // persistent kernels: exactly as many CTAs as can be resident (one wave), so every CTA pulls work until the pass is drained
  // (the inline scene's kernels are instantiated here first, in this order: ptxas output depends on the module's entry order)
  RaynContext::Occ& o = ctx->occ[0];
  for (int v = 0; v < SDFV_COUNT && e == cudaSuccess; ++v) {
    DISPATCH_SDFV(v, e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.ext[v], k_extend_march<V, DevScene>, EXT_T, 0);
                  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.shd[v], k_shadow<V, DevScene>, SHD_T, 0);
                  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.nrm[v], k_normals<V, DevScene>, SLOT_BLOCK, 0));
  }
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.pre, k_shade_pre<DevScene>, SLOT_BLOCK, 0);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.post, k_shade_post<DevScene>, SLOT_BLOCK, 0);
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.sph, k_extend_spheres<DevScene>, EXT_BATCH, 0);
  if (e == cudaSuccess) e = query_occupancy<TableScene>(ctx->occ[1]);
  if (e != cudaSuccess) {
    cudaGetLastError();
    fail(nullptr, RAYN_ERR_CUDA, "context setup: %s", cudaGetErrorString(e));
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    cudaFree(ctx->pb.counters), cudaFree(ctx->d_fis), cudaFree(ctx->d_work_ctr), cudaFree(ctx->d_kat);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    delete ctx;
    return RAYN_ERR_CUDA;
  }
  *out_ctx = ctx;
  return RAYN_OK;
}

int32_t rayn_b200_comm_destroy(RaynContext* ctx) {
  if (!ctx) return RAYN_ERR_INVALID_ARG;
  RaynComm& c = ctx->comm;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (c.comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c.comm);
  cudaFree(c.d_table), cudaFree(c.d_slabs);
  c = RaynComm();
  return RAYN_OK;
}

void rayn_b200_destroy(RaynContext* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  rayn_b200_comm_destroy(ctx);
  free_pass(ctx);
  cudaFree(ctx->pb.counters);
  cudaFree(ctx->d_work_ctr);
  cudaFree(ctx->d_kat);
  cudaFree(ctx->d_pack_ids);
  cudaFree(ctx->d_post);
  cudaFree(ctx->d_s1), cudaFree(ctx->d_s2), cudaFree(ctx->d_scr), cudaFree(ctx->d_fis), cudaFree(ctx->d_planes);
  cudaFree(ctx->d_tables);
  for (auto& t : ctx->timed) cudaEventDestroy(t.a), cudaEventDestroy(t.b);
  if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
  cudaEventDestroy(ctx->ev0), cudaEventDestroy(ctx->ev1);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

static int32_t validate_scene(RaynContext* ctx, const RaynSceneDesc* s) {
  if (!s) return fail(ctx, RAYN_ERR_INVALID_ARG, "scene is NULL");
  if (s->n_hitables < 1 || s->n_hitables > RAYN_MAX_HITABLES)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "n_hitables %d not in [1,%d] (RAYN_MAX_HITABLES)", s->n_hitables, RAYN_MAX_HITABLES);
  if (s->n_materials < 1 || s->n_materials > RAYN_MAX_MATERIALS)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "n_materials %d not in [1,%d] (RAYN_MAX_MATERIALS)", s->n_materials, RAYN_MAX_MATERIALS);
  if (s->n_lights < 0 || s->n_lights > RAYN_MAX_LIGHTS)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "n_lights %d not in [0,%d] (RAYN_MAX_LIGHTS)", s->n_lights, RAYN_MAX_LIGHTS);
  if (!s->hitables || !s->materials || (s->n_lights && !s->lights)) return fail(ctx, RAYN_ERR_INVALID_ARG, "NULL scene array");
  int n_sdf = 0;
  for (int i = 0; i < s->n_hitables; ++i) n_sdf += s->hitables[i].kind != RAYN_HITABLE_SPHERE ? 1 : 0;
  if (n_sdf > RAYN_MAX_SDF_HITABLES)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "%d SDF hitables, more than %d (RAYN_MAX_SDF_HITABLES)", n_sdf, RAYN_MAX_SDF_HITABLES);
  for (int i = 0; i < s->n_hitables; ++i) {
    const RaynHitable& h = s->hitables[i];
    if (h.kind < 0 || h.kind > RAYN_HITABLE_MANDELBULB) return fail(ctx, RAYN_ERR_INVALID_ARG, "hitable %d: bad kind %d", i, h.kind);
    if (h.material < 0 || h.material >= s->n_materials)
      return fail(ctx, RAYN_ERR_INVALID_ARG, "hitable %d: material %d out of range", i, h.material);
    if (h.kind != RAYN_HITABLE_SPHERE && (h.iterations < 0 || h.iterations > 1024))
      return fail(ctx, RAYN_ERR_INVALID_ARG, "hitable %d: iterations %d", i, h.iterations);
    if (h.kind == RAYN_HITABLE_MANDELBULB && h.bulb_power != 8)
      return fail(ctx, RAYN_ERR_UNSUPPORTED, "hitable %d: Mandelbulb power %d (only 8 is built)", i, h.bulb_power);
  }
  for (int i = 0; i < s->n_materials; ++i)
    if (s->materials[i].kind < 0 || s->materials[i].kind > RAYN_MATERIAL_EMISSIVE)
      return fail(ctx, RAYN_ERR_INVALID_ARG, "material %d: bad kind %d", i, s->materials[i].kind);
  if (s->camera.kind < 0 || s->camera.kind > RAYN_CAMERA_ORTHOGRAPHIC) return fail(ctx, RAYN_ERR_INVALID_ARG, "bad camera kind");
  if (s->consts.max_marches < 1 || s->consts.max_vis_marches < 1) return fail(ctx, RAYN_ERR_INVALID_ARG, "march limits must be >= 1");
  return RAYN_OK;
}

// Is the three-operation sphere-fold division (rt_sdf2.cuh::fastdiv2_3) equal to IEEE division for EVERY divisor this
// Mandelbox can produce?  The divisor is clamp(r2, min_r2, fixed_r2), so the candidates are the floats of that interval: all of
// them are divided on the device, once per (min_r2, fixed_r2) pair and context (~0.1 ms per 10^8 divisors).
static bool div3_verified(RaynContext* ctx, const RaynHitable& h) {
  if (!sdf_box_fast_ok(h)) return false;
  for (const auto& c : ctx->div3_cache)
    if (c.min_r2 == h.min_rad_sq && c.fixed_r2 == h.fixed_rad_sq) return c.ok;
  bool ok = false;
  uint32_t lo, hi;
  memcpy(&lo, &h.min_rad_sq, 4);
  memcpy(&hi, &h.fixed_rad_sq, 4);
  if (hi >= lo && cudaSetDevice(ctx->device) == cudaSuccess) {  // positive floats order like their bit patterns
    const unsigned long long n = (unsigned long long)(hi - lo) + 1ull;
    unsigned long long bad = 1;
    if (cudaMemsetAsync(ctx->d_kat, 0, sizeof(unsigned long long), ctx->stream) == cudaSuccess) {
      k_verify_div3<<<ctx->n_sm * 8, 256, 0, ctx->stream>>>(h.fixed_rad_sq, lo, n, ctx->d_kat);
      if (cudaMemcpyAsync(&bad, ctx->d_kat, sizeof bad, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess &&
          cudaStreamSynchronize(ctx->stream) == cudaSuccess)
        ok = bad == 0;
    }
    cudaGetLastError();
  }
  ctx->div3_cache.push_back({h.min_rad_sq, h.fixed_rad_sq, ok});
  return ok;
}

int32_t rayn_b200_upload_scene(RaynContext* ctx, const RaynSceneDesc* s) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  int32_t rc = validate_scene(ctx, s);
  if (rc) return rc;
  ctx->has_scene = false;
  const int nh = s->n_hitables, nm = s->n_materials, nl = s->n_lights;
  ctx->h_hit.assign(s->hitables, s->hitables + nh);
  ctx->h_mat.assign(s->materials, s->materials + nm);
  // compact sphere / SDF lists in insertion order (DevScene)
  std::vector<int32_t> sph_idx, sdf_idx, hit_ord(nh);
  std::vector<float4> sph;
  int sph_moving = 0;
  for (int i = 0; i < nh; ++i) {
    const RaynHitable& h = s->hitables[i];
    if (h.kind == RAYN_HITABLE_SPHERE) {
      hit_ord[i] = (int32_t)sph_idx.size();
      sph_idx.push_back(i);
      sph.push_back(make_float4(h.center[0], h.center[1], h.center[2], h.radius));
      sph_moving |= (h.center_velocity[0] != 0.0f || h.center_velocity[1] != 0.0f || h.center_velocity[2] != 0.0f) ? 1 : 0;
    } else {
      hit_ord[i] = (int32_t)sdf_idx.size();
      sdf_idx.push_back(i);
    }
  }
  DevScene& d = ctx->scene;
  memset(&d, 0, sizeof d);
  d.n_hit = nh;
  d.n_mat = nm;
  d.n_lights = nl;
  d.one = 1.0f;
  d.cam = s->camera;
  d.vol = s->volume;
  d.rc = s->consts;
  d.n_sph = (int32_t)sph_idx.size();
  d.n_sdf = (int32_t)sdf_idx.size();
  d.sph_moving = sph_moving;
  ctx->tables = (ctx->flags & RAYN_FLAG_SCENE_TABLES) || nh > SCENE_INLINE_MAX || nm > SCENE_INLINE_MAX || nl > SCENE_INLINE_MAX;
  if (!ctx->tables) {
    memcpy(d.hit, s->hitables, sizeof(RaynHitable) * nh);
    memcpy(d.mat, s->materials, sizeof(RaynMaterial) * nm);
    if (nl) memcpy(d.light, s->lights, sizeof(RaynLight) * nl);
    std::copy(sph_idx.begin(), sph_idx.end(), d.sph_idx);
    std::copy(sdf_idx.begin(), sdf_idx.end(), d.sdf_idx);
    std::copy(hit_ord.begin(), hit_ord.end(), d.hit_ord);
    std::copy(sph.begin(), sph.end(), d.sph);
  } else {
    // one device block: the seven tables, each 256-byte aligned
    size_t off[7], total = 0;
    const size_t bytes[7] = {sizeof(RaynHitable) * nh, sizeof(RaynMaterial) * nm, sizeof(RaynLight) * nl, sizeof(int32_t) * sph_idx.size(),
                             sizeof(int32_t) * sdf_idx.size(), sizeof(int32_t) * nh, sizeof(float4) * sph.size()};
    const void* src[7] = {s->hitables, s->materials, s->lights, sph_idx.data(), sdf_idx.data(), hit_ord.data(), sph.data()};
    for (int t = 0; t < 7; ++t) off[t] = total, total += (bytes[t] + 255) & ~(size_t)255;
    std::vector<unsigned char> blob(total, 0);
    for (int t = 0; t < 7; ++t)
      if (bytes[t]) memcpy(blob.data() + off[t], src[t], bytes[t]);
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));  // kernels still in flight may read the tables that are rewritten here
    CU(regrow(&ctx->d_tables, &ctx->cap_tables, total));
    CU(cudaMemcpyAsync(ctx->d_tables, blob.data(), total, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    TableScene& t = ctx->tscene;
    memset(&t, 0, sizeof t);
    t.n_hit = d.n_hit, t.n_mat = d.n_mat, t.n_lights = d.n_lights, t.one = d.one;
    t.hit.p = (const RaynHitable*)(ctx->d_tables + off[0]);
    t.mat.p = (const RaynMaterial*)(ctx->d_tables + off[1]);
    t.light.p = (const RaynLight*)(ctx->d_tables + off[2]);
    t.cam = d.cam, t.vol = d.vol, t.rc = d.rc;
    t.n_sph = d.n_sph, t.n_sdf = d.n_sdf, t.sph_moving = d.sph_moving;
    t.sph_idx.p = (const int32_t*)(ctx->d_tables + off[3]);
    t.sdf_idx.p = (const int32_t*)(ctx->d_tables + off[4]);
    t.hit_ord.p = (const int32_t*)(ctx->d_tables + off[5]);
    t.sph.p = (const float4*)(ctx->d_tables + off[6]);
  }
  ++ctx->scene_gen;
  for (int i = 0; i < nh; ++i)
    ctx->sdf_var[i] = s->hitables[i].kind == RAYN_HITABLE_SPHERE ? -1 : sdf_variant(s->hitables[i], !(ctx->flags & RAYN_FLAG_NO_DIV3) && div3_verified(ctx, s->hitables[i]));
  ctx->has_scene = true;
  return RAYN_OK;
}

int32_t rayn_b200_get_stats(const RaynContext* ctx, RaynStats* out) {
  if (!ctx || !out) return RAYN_ERR_INVALID_ARG;
  *out = ctx->stats;
  return RAYN_OK;
}

int32_t rayn_b200_debug_sdf_variant(const RaynContext* ctx, int32_t hitable_index) {
  if (!ctx || !ctx->has_scene || hitable_index < 0 || hitable_index >= ctx->scene.n_hit) return -2;
  return ctx->sdf_var[hitable_index];
}

int32_t rayn_b200_debug_enable_queue_log(RaynContext* ctx, int32_t enable) {
  if (!ctx) return RAYN_ERR_INVALID_ARG;
  ctx->qlog_enabled = enable != 0;
  ctx->qlog.clear();
  return RAYN_OK;
}
int64_t rayn_b200_debug_read_queue_log(RaynContext* ctx, int32_t* out, int64_t cap) {
  if (!ctx) return -1;
  const int64_t n = (int64_t)ctx->qlog.size();
  if (out && cap > 0) memcpy(out, ctx->qlog.data(), sizeof(int32_t) * (size_t)std::min(n, cap));
  return n;
}

}  // extern "C"

// Enqueues one render on the context's stream.  Nothing here waits for the GPU (except the debug queue log), so a single
// host thread can keep several GPUs busy (render_frame_multi).  tiles_override replaces the frame's own tile selection.
// dev_planes_out (optional) receives the device-space planes the film was rendered into.
static int32_t render_enqueue(RaynContext* ctx, const RaynFrameDesc* f, const RaynFilmPlanes* out, const std::vector<int>* tiles_override,
                              RaynFilmPlanes* dev_planes_out) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  if (ctx->pending) return fail(ctx, RAYN_ERR_INVALID_ARG, "a render is already in flight on this context");
  if (!ctx->has_scene) return fail(ctx, RAYN_ERR_NO_SCENE, "render_frame before upload_scene");
  if (!f || !out) return fail(ctx, RAYN_ERR_INVALID_ARG, "frame/out is NULL");
  if (f->width <= 0 || f->height <= 0 || f->tile_w <= 0 || f->tile_h <= 0 || f->samples <= 0 || f->max_bounces < 0)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "bad frame geometry");
  if (f->volume_marches != 2)
    return fail(ctx, RAYN_ERR_UNSUPPORTED, "volume_marches = %d: the reference hard-wires samples_1d[3],[4] for vm = 2", f->volume_marches);
  const int spp = 4 * f->samples, vm = f->volume_marches, mb = f->max_bounces;
  const int need1 = 1 + (mb + 1) * (3 + vm), need2 = 2 + (mb + 1) * (12 + 8 * vm) / 2;
  if (f->sets_1d < need1 || f->sets_2d < need2)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "sample tables too small: have %d/%d sets, path needs %d/%d", f->sets_1d, f->sets_2d, need1, need2);
  if (!f->samples_1d || !f->samples_2d || !f->scramble || !f->fis_inverse_cdf) return fail(ctx, RAYN_ERR_INVALID_ARG, "NULL input table");
  const int stride = f->tile_stride > 0 ? f->tile_stride : 1;
  if (!tiles_override && !f->tile_list && (f->tile_offset < 0 || f->tile_offset >= stride))
    return fail(ctx, RAYN_ERR_INVALID_ARG, "tile_offset %d not in [0,%d)", f->tile_offset, stride);
  if (mb >= TERM_MAX_DEPTH) return fail(ctx, RAYN_ERR_UNSUPPORTED, "max_bounces > %d", TERM_MAX_DEPTH - 1);
  const int64_t R64 = (int64_t)f->tile_w * f->tile_h * spp;
  const int n_hit = ctx->scene.n_hit;
  if (R64 + 4 * n_hit >= TERM_MAX_SLOTS)
    return fail(ctx, RAYN_ERR_UNSUPPORTED, "tile_w*tile_h*spp = %lld exceeds the 2^%d slot key space", (long long)R64, TERM_DEPTH_SHIFT);
  int np = 32;
  while (np < spp) np <<= 1;
  const int wpc = resolve_warps_per_cta(np);
  if (wpc < 1 || np > 65536) return fail(ctx, RAYN_ERR_UNSUPPORTED, "spp = %d: the film resolve holds 6 B per sample of a pixel in shared memory (max 32768 spp)", spp);
  const int R = (int)R64, QS = R + 4 * n_hit;
  CU(cudaSetDevice(ctx->device));
  {  // a previous call that failed half way through a graph capture must not leave the stream capturing
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(ctx->stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
      cudaGraph_t g = nullptr;
      cudaStreamEndCapture(ctx->stream, &g);
      if (g) cudaGraphDestroy(g);
    }
    cudaGetLastError();
  }

  DevFrame fr;
  fr.W = f->width, fr.H = f->height, fr.tile_w = f->tile_w, fr.tile_h = f->tile_h;
  fr.samples = f->samples, fr.spp = spp, fr.max_bounces = mb, fr.vm = vm;
  tile_grid_of(f->width, f->height, f->tile_w, f->tile_h, &fr.ntx, &fr.nty);
  fr.sets_1d = f->sets_1d, fr.sets_2d = f->sets_2d;
  fr.t0 = f->t0, fr.t1 = f->t1;

  std::vector<int>& my_tiles = ctx->job_tiles;
  my_tiles.clear();
  if (tiles_override) {
    my_tiles = *tiles_override;
  } else if (f->tile_list) {
    if (f->n_tile_list < 0) return fail(ctx, RAYN_ERR_INVALID_ARG, "n_tile_list < 0");
    for (int i = 0; i < f->n_tile_list; ++i) {
      const int idx = f->tile_list[i];
      if (idx < 0 || idx >= fr.ntx * fr.nty || (i && idx <= f->tile_list[i - 1]))
        return fail(ctx, RAYN_ERR_INVALID_ARG, "tile_list must be ascending tile indices in [0,%d)", fr.ntx * fr.nty);
      my_tiles.push_back(idx);
    }
  } else {
    for (int idx = f->tile_offset; idx < fr.ntx * fr.nty; idx += stride) my_tiles.push_back(idx);
  }

  memset(&ctx->stats, 0, sizeof ctx->stats);
  ctx->timed_used = 0;
  ctx->qlog.clear();
  cudaStream_t st = ctx->stream;

  // Device-space pointers may have been produced on another stream (e.g. torch's): fence.
  if (f->input_space == RAYN_MEM_DEVICE || out->space == RAYN_MEM_DEVICE) CU(cudaDeviceSynchronize());
  CU(cudaEventRecord(ctx->ev0, st));

  const size_t n1 = (size_t)spp * f->sets_1d, n2 = (size_t)2 * spp * f->sets_2d, npx = (size_t)f->width * f->height;
  if (f->input_space == RAYN_MEM_HOST) {
    CU(regrow(&ctx->d_s1, &ctx->cap_s1, n1));
    CU(regrow(&ctx->d_s2, &ctx->cap_s2, n2));
    CU(regrow(&ctx->d_scr, &ctx->cap_scr, npx));
    CU(cudaMemcpyAsync(ctx->d_s1, f->samples_1d, n1 * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_s2, f->samples_2d, n2 * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_scr, f->scramble, npx * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_fis, f->fis_inverse_cdf, RAYN_FIS_TABLE_SIZE * 4, cudaMemcpyHostToDevice, st));
    fr.s1 = ctx->d_s1, fr.s2 = ctx->d_s2, fr.scramble = ctx->d_scr, fr.fis = ctx->d_fis;
  } else {
    fr.s1 = f->samples_1d, fr.s2 = f->samples_2d, fr.scramble = f->scramble, fr.fis = f->fis_inverse_cdf;
  }
  float *p_color, *p_alpha, *p_bg, *p_normal;
  if (out->space == RAYN_MEM_HOST) {
    CU(regrow(&ctx->d_planes, &ctx->cap_planes, npx * 10));
    CU(cudaMemsetAsync(ctx->d_planes, 0, npx * 10 * 4, st));
    p_color = ctx->d_planes, p_alpha = p_color + 3 * npx, p_bg = p_alpha + npx, p_normal = p_bg + 3 * npx;
  } else {
    p_color = out->color, p_alpha = out->alpha, p_bg = out->background, p_normal = out->normal;
    const int cov_w = std::min(fr.ntx * f->tile_w, f->width), cov_h = std::min(fr.nty * f->tile_h, f->height);
    if (cov_w < f->width || cov_h < f->height)
      k_zero_uncovered<<<(unsigned)((npx + 255) / 256), 256, 0, st>>>(f->width, f->height, cov_w, cov_h, p_color, p_alpha, p_bg, p_normal);
  }
  if (dev_planes_out) {
    dev_planes_out->color = p_color, dev_planes_out->alpha = p_alpha, dev_planes_out->background = p_bg, dev_planes_out->normal = p_normal;
    dev_planes_out->space = RAYN_MEM_DEVICE;
  }

  const std::vector<RaynHitable>& hit = ctx->h_hit;
  std::vector<int> sdf_idx;
  for (int i = 0; i < n_hit; ++i)
    if (hit[i].kind != RAYN_HITABLE_SPHERE) sdf_idx.push_back(i);
  const int n_sdf = (int)sdf_idx.size();
  const bool simple = (ctx->flags & RAYN_FLAG_SIMPLE_MARCH) != 0;
  if (simple && ctx->tables)
    return fail(ctx, RAYN_ERR_UNSUPPORTED, "scenes beyond %d hitables, materials or lights are not supported by the legacy test kernels", SCENE_INLINE_MAX);
  bool motion = false;  // time-varying sphere centres need the packet's lane-0 time: only the product kernels plumb it
  for (int i = 0; i < n_hit; ++i)
    motion |= hit[i].kind == RAYN_HITABLE_SPHERE && (hit[i].center_velocity[0] != 0.0f || hit[i].center_velocity[1] != 0.0f || hit[i].center_velocity[2] != 0.0f);
  if (motion && simple) return fail(ctx, RAYN_ERR_UNSUPPORTED, "time-varying sphere centres are not supported by the legacy test kernels");
  // leading analytic spheres run inside raygen / shade_post (rt_kernels.cuh::fold_head); -1 = not folded (moving spheres need
  // the extend packet's lane-0 time; the legacy test kernels do the whole fold themselves)
  int fold_pre = -1;
  if (!motion && !simple) {
    fold_pre = 0;
    while (fold_pre < n_hit && hit[fold_pre].kind == RAYN_HITABLE_SPHERE) ++fold_pre;
  }
  // Scenes of the shape [spheres] Mandelbox [spheres] (setup.rs) fold ALL analytic spheres into the producing kernel and march
  // the SDF last, against the nearest sphere: one gather of every live ray per depth less (k_extend_spheres was 2 % of a
  // config-3 frame) and shorter marches for rays that end on an emitter.  The result is the reference's fold bit for bit
  // (proof in rt_kernels.cuh at k_extend_march: it needs a distance estimator that is never negative, i.e. the Mandelbox -
  // sqrt(m) / |dr| - so that a march's t never decreases, and the first-index-wins tie rule, which the kernel applies).
  const bool fold_all = fold_pre >= 0 && n_sdf == 1 && hit[sdf_idx[0]].kind == RAYN_HITABLE_MANDELBOX && !(ctx->flags & RAYN_FLAG_NO_FOLD_ALL);
  const int n_fold = fold_all ? ctx->scene.n_sph : fold_pre;  // leading spheres are the first fold_pre entries of the compact sphere list
  const bool volume_on = ctx->scene.vol.has_scattering != 0 && ctx->scene.n_lights > 0;
  const int ns = volume_on ? 4 * (1 + vm) : 4;               // light samples per path per depth
  const int seg_per_path = simple ? 0 : ns * n_sdf;          // worst case shadow segments per path per depth, all SDF queues
  const int lc_ns = simple ? 0 : ns;                         // stored light contributions per path per depth
  const int maxk = ctx->tables ? TableScene::kMaxHit : DevScene::kMaxHit;  // keys of the bin kernels, row stride of the bin tables
  const RaynContext::Occ& occ = ctx->occ[ctx->tables ? 1 : 0];

  // pass size: as many tiles as the requested path budget AND free device memory allow
  const size_t bpp = pass_bytes_per_path(R, QS, seg_per_path, lc_ns, maxk);
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  const size_t budget = (size_t)((double)(free_b + ctx->pass_bytes) * 0.90);
  int64_t max_paths = std::min<int64_t>(ctx->cap_paths, (int64_t)(budget / bpp));
  if (n_sdf > 0) max_paths = std::min<int64_t>(max_paths, ((int64_t)1 << 27) - 1);          // owner path index is packed with the sample bit (<< 4)
  if (n_sdf > 0) max_paths = std::min<int64_t>(max_paths, (int64_t)INT_MAX / std::max(ns, 1));  // 32-bit queue cursors per SDF
  int tiles_per_pass = (int)std::max<int64_t>(1, max_paths / R);
  tiles_per_pass = std::min(tiles_per_pass, 65535);
  tiles_per_pass = std::min<int>(tiles_per_pass, (int)std::max<size_t>(my_tiles.size(), 1));
  int32_t rc;
  while ((rc = ensure_pass(ctx, tiles_per_pass, R, QS, seg_per_path, n_sdf, lc_ns, maxk)) == RAYN_ERR_OOM && tiles_per_pass > 1)
    tiles_per_pass = (tiles_per_pass + 1) / 2;  // fragmentation / another tenant: retry with half the pass
  if (rc) return rc;
  PassBufs pb = ctx->pb;
  pb.R = R, pb.QS = QS, pb.tile_ids = ctx->d_tile_ids;
  pb.lc_ns = lc_ns;
  pb.seg_count = ctx->d_work_ctr + WC_SEG_COUNT;
  CU(cudaMemsetAsync(pb.counters, 0, CNT_TOTAL * sizeof(unsigned long long), st));
  const size_t res_smem = resolve_smem_per_warp(np) * wpc;
  int slot_bits = 5, depth_bits = 1;  // significant bits of a shading slot (< QS) and of a depth (<= max_bounces): what k_resolve's radix sort walks
  while ((1 << slot_bits) < QS + 1) ++slot_bits;
  while ((1 << depth_bits) < mb + 1) ++depth_bits;
  CU(cudaFuncSetAttribute(k_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)res_smem));

  // Small single-pass frames are launch bound (config 1: ~20 launches of a few microseconds each): capture the whole kernel
  // sequence of the pass once and replay it as ONE graph launch while nothing that is baked into the launches changes
  // (scene, frame geometry, every pointer, the tile set).
  const bool single_pass = my_tiles.size() <= (size_t)tiles_per_pass;
  const bool use_graph = single_pass && !my_tiles.empty() && !(ctx->flags & (RAYN_FLAG_TIMING | RAYN_FLAG_NO_GRAPH)) && !ctx->qlog_enabled &&
                         (int64_t)my_tiles.size() * R <= ((int64_t)8 << 20);
  bool capturing = false, replayed = false;
  uint64_t key = 0;
  if (use_graph) {
    PassBufs kpb = pb;
    kpb.n_tiles = (int)my_tiles.size();
    key = fnv1a(1469598103934665603ull, &ctx->scene, sizeof ctx->scene);
    if (ctx->tables) {  // the launches carry only the tables' pointers: the upload count stands for their contents
      key = fnv1a(key, &ctx->tscene, sizeof ctx->tscene);
      key = fnv1a(key, &ctx->scene_gen, sizeof ctx->scene_gen);
    }
    key = fnv1a(key, &fr, sizeof fr);
    key = fnv1a(key, &kpb, sizeof kpb);
    float* planes4[4] = {p_color, p_alpha, p_bg, p_normal};
    key = fnv1a(key, planes4, sizeof planes4);
    const int misc[6] = {np, wpc, mb, n_fold, simple ? 1 : 0, motion ? 1 : 0};
    key = fnv1a(key, misc, sizeof misc);
    key = fnv1a(key, my_tiles.data(), my_tiles.size() * sizeof(int));
    if (ctx->graph_exec && ctx->graph_key == key) {
      CU(cudaMemcpyAsync(ctx->d_tile_ids, my_tiles.data(), my_tiles.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      CU(cudaGraphLaunch(ctx->graph_exec, st));
      ctx->stats = ctx->graph_stats;
      replayed = true;
    }
  }
  std::vector<int> h_nslots, h_slots;
  // the kernel sequence of one pass of nt tiles starting at my_tiles[first], for either scene type
  auto run_pass = [&](const auto& sc, const int nt, const size_t first) -> int32_t {
    using S = std::decay_t<decltype(sc)>;
    const dim3 g_paths((R + 255) / 256, nt), g_shade((QS + 127) / 128, nt);
    (void)g_shade;
    // resident grids (one wave) of the kernels that stride over a work list (k_scan_slots / k_scan_live), capped by the list's upper bound
    const int64_t max_blocks = (int64_t)nt * ((QS + SLOT_BLOCK - 1) / SLOT_BLOCK);
    auto resident = [&](int o) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>((int64_t)ctx->n_sm * o, max_blocks)); };
    const int nseg = (QS + SEG_SLOTS - 1) / SEG_SLOTS;  // segments per tile of the queue kernels
    timed_begin(ctx, RAYN_K_RAYGEN);
    k_raygen<S><<<g_paths, 256, 0, st>>>(sc, fr, pb, n_fold);
    timed_end(ctx, RAYN_K_RAYGEN);
    for (int depth = 0; depth <= mb; ++depth) {
      const Thr thr = make_thr(ctx->scene.cam, depth);
      if (simple) {
#ifdef RAYN_LEGACY_KERNELS
        timed_begin(ctx, RAYN_K_EXTEND);
        k_extend<<<dim3((R + 127) / 128, nt), 128, 0, st>>>(ctx->scene, pb, thr);
        timed_end(ctx, RAYN_K_EXTEND);
#endif
      } else {
        timed_begin(ctx, RAYN_K_MISC);
        k_scan_live<<<1, SCAN_T, 0, st>>>(pb, ctx->d_batch_prefix, ctx->d_work_ctr);
        timed_end(ctx, RAYN_K_MISC);
        // fold order of hitable.rs:177-198: runs of spheres as coherent kernels, each SDF as a persistent march.  The
        // spheres before the first SDF were already folded in by the kernel that produced the rays (fold_pre >= 0).
        int k = fold_pre >= 0 ? fold_pre : 0, first_kernel = fold_pre >= 0 ? 0 : 1, n_march = 0;
        while (k < n_hit || first_kernel) {
          int e = k;
          while (e < n_hit && hit[e].kind == RAYN_HITABLE_SPHERE) ++e;
          if ((e > k || first_kernel) && !fold_all) {
            const int run = (int)(std::lower_bound(sdf_idx.begin(), sdf_idx.end(), k) - sdf_idx.begin());  // SDFs before the run
            timed_begin(ctx, RAYN_K_EXTEND_SPHERES);
            k_extend_spheres<S><<<resident(occ.sph), EXT_BATCH, 0, st>>>(sc, pb, k, e, first_kernel, motion ? 1 : 0, ctx->d_batch_prefix, ctx->d_work_ctr + WC_SPHERES + run);
            timed_end(ctx, RAYN_K_EXTEND_SPHERES);
            first_kernel = 0;
          }
          if (e < n_hit) {
            if (n_march++ > 0) CU(cudaMemsetAsync(ctx->d_work_ctr + WC_EXTEND, 0, sizeof(int), st));
            const int v = ctx->sdf_var[e];
            timed_begin(ctx, RAYN_K_EXTEND);
            DISPATCH_SDFV(v, (k_extend_march<V, S><<<ctx->n_sm * occ.ext[v], EXT_T, 0, st>>>(sc, pb, thr, e, fold_all ? 1 : 0, ctx->d_batch_prefix, ctx->d_work_ctr + WC_EXTEND)));
            timed_end(ctx, RAYN_K_EXTEND);
            ++e;
          }
          k = e;
        }
      }
      timed_begin(ctx, RAYN_K_BIN);
      k_bin_count<S::kMaxHit><<<dim3(nseg, nt), BIN_T, 0, st>>>(pb, n_hit, nseg);
      if (ctx->tables)
        k_bin_scatter_tables<<<dim3(nseg, nt), BINB_T, 0, st>>>(pb, n_hit, nseg);
      else
        k_bin_scatter<<<dim3(nseg, nt), BIN_T, 0, st>>>(pb, n_hit, nseg);
      if (!simple) k_scan_slots<S><<<1, SCAN_T, 0, st>>>(sc, pb);  // work lists of k_normals / k_shade_pre / k_shade_post
      timed_end(ctx, RAYN_K_BIN, simple ? 2 : 3);
      if (ctx->qlog_enabled) {
        h_nslots.resize(nt);
        h_slots.resize((size_t)nt * QS);
        CU(cudaMemcpyAsync(h_nslots.data(), pb.n_slots, nt * sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h_slots.data(), pb.q_shade, (size_t)nt * QS * sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (int t = 0; t < nt; ++t) {
          ctx->qlog.push_back(depth);
          ctx->qlog.push_back(my_tiles[first + t]);
          ctx->qlog.push_back(h_nslots[t]);
          for (int s = 0; s < h_nslots[t]; ++s) ctx->qlog.push_back(h_slots[(size_t)t * QS + s]);
        }
      }
      if (!simple) {
        // get_shading_info of the SDF hitables whose material is shaded (receives light, or volumetrics sample along the ray)
        for (int j = 0; j < n_sdf; ++j) {
          const RaynHitable& h = hit[sdf_idx[j]];
          const int mk = ctx->h_mat[h.material].kind;
          if (!(mk == RAYN_MATERIAL_LAMBERTIAN || mk == RAYN_MATERIAL_DIELECTRIC || volume_on)) continue;
          const int v = ctx->sdf_var[sdf_idx[j]];
          timed_begin(ctx, RAYN_K_NORMALS);
          DISPATCH_SDFV(v, (k_normals<V, S><<<resident(occ.nrm[v]), SLOT_BLOCK, 0, st>>>(sc, pb, thr, sdf_idx[j], j, ctx->d_work_ctr + WC_NORMALS + j)));
          timed_end(ctx, RAYN_K_NORMALS);
        }
        timed_begin(ctx, RAYN_K_SHADE_PRE);
        k_shade_pre<S><<<resident(occ.pre), SLOT_BLOCK, 0, st>>>(sc, fr, pb, depth, thr, ctx->d_work_ctr + WC_PRE);
        timed_end(ctx, RAYN_K_SHADE_PRE);
        if (ctx->scene.n_lights > 0) {
          for (int j = 0; j < n_sdf; ++j) {
            const int v = ctx->sdf_var[sdf_idx[j]];
            timed_begin(ctx, RAYN_K_SHADOW);
            DISPATCH_SDFV(v, (k_shadow<V, S><<<ctx->n_sm * occ.shd[v], SHD_T, 0, st>>>(sc, pb, sdf_idx[j], j, ctx->d_work_ctr + WC_SHADOW + j)));
            timed_end(ctx, RAYN_K_SHADOW);
          }
        }
        timed_begin(ctx, RAYN_K_SHADE_POST);
        k_shade_post<S><<<resident(occ.post), SLOT_BLOCK, 0, st>>>(sc, fr, pb, depth, n_fold, ctx->d_work_ctr + WC_POST);
        timed_end(ctx, RAYN_K_SHADE_POST);
      } else {
#ifdef RAYN_LEGACY_KERNELS
        timed_begin(ctx, RAYN_K_SHADE_PRE);
        k_shade<<<g_shade, 128, 0, st>>>(ctx->scene, fr, pb, depth, thr);
        timed_end(ctx, RAYN_K_SHADE_PRE);
#endif
      }
      if (depth < mb) {
        timed_begin(ctx, RAYN_K_COMPACT);
        k_compact_count<<<dim3(nseg, nt), CMP_T, 0, st>>>(pb, nseg);
        k_compact_scatter<<<dim3(nseg, nt), CMP_T, 0, st>>>(pb, nseg);
        timed_end(ctx, RAYN_K_COMPACT, 2);
      }
    }
    timed_begin(ctx, RAYN_K_RESOLVE);
    k_resolve<<<dim3((f->tile_w * f->tile_h + wpc - 1) / wpc, nt), wpc * 32, res_smem, st>>>(fr, pb, p_color, p_alpha, p_bg, p_normal, np, wpc, slot_bits, depth_bits);
    timed_end(ctx, RAYN_K_RESOLVE);
    return RAYN_OK;
  };
  for (size_t first = 0; first < my_tiles.size() && !replayed; first += tiles_per_pass) {
    const int nt = (int)std::min<size_t>(tiles_per_pass, my_tiles.size() - first);
    pb.n_tiles = nt;
    CU(cudaMemcpyAsync(ctx->d_tile_ids, my_tiles.data() + first, nt * sizeof(int), cudaMemcpyHostToDevice, st));
    if (use_graph) {
      CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      capturing = true;
    }
    ctx->stats.passes++;
    if ((rc = ctx->tables ? run_pass(ctx->tscene, nt, first) : run_pass(ctx->scene, nt, first))) return rc;
    if (capturing) {
      cudaGraph_t graph = nullptr;
      CU(cudaStreamEndCapture(st, &graph));
      capturing = false;
      if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
      ctx->graph_exec = nullptr;
      const cudaError_t ge = cudaGraphInstantiate(&ctx->graph_exec, graph, 0);
      cudaGraphDestroy(graph);
      CU(ge);
      ctx->graph_key = key;
      ctx->graph_stats = ctx->stats;
      ctx->graph_stats.reserved_ = 1;  // marks "replayed from a captured graph" for callers that look
      CU(cudaGraphLaunch(ctx->graph_exec, st));
      ctx->stats.reserved_ = 1;  // this frame, too, ran as one graph launch
    }
    CU(cudaGetLastError());
  }
  ctx->job_w = f->width, ctx->job_h = f->height, ctx->job_tw = f->tile_w, ctx->job_th = f->tile_h, ctx->job_spp = spp, ctx->job_nty = fr.nty;
  ctx->pending = true;
  return RAYN_OK;
}

// D2H of host-space planes (after an optional gather), then the end-of-frame bookkeeping
static int32_t copy_out_enqueue(RaynContext* ctx, const RaynFilmPlanes* out) {
  if (out->space != RAYN_MEM_HOST) return RAYN_OK;
  cudaStream_t st = ctx->stream;
  const size_t npx = (size_t)ctx->job_w * ctx->job_h;
  const float* d = ctx->d_planes;
  if (out->color) CU(cudaMemcpyAsync(out->color, d, npx * 3 * 4, cudaMemcpyDeviceToHost, st));
  if (out->alpha) CU(cudaMemcpyAsync(out->alpha, d + 3 * npx, npx * 4, cudaMemcpyDeviceToHost, st));
  if (out->background) CU(cudaMemcpyAsync(out->background, d + 4 * npx, npx * 3 * 4, cudaMemcpyDeviceToHost, st));
  if (out->normal) CU(cudaMemcpyAsync(out->normal, d + 7 * npx, npx * 3 * 4, cudaMemcpyDeviceToHost, st));
  return RAYN_OK;
}

static int32_t render_finish(RaynContext* ctx) {
  if (!ctx->pending) return RAYN_OK;
  ctx->pending = false;
  cudaStream_t st = ctx->stream;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventRecord(ctx->ev1, st));
  CU(cudaMemcpyAsync(ctx->h_counters, ctx->pb.counters, sizeof ctx->h_counters, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  CU(cudaGetLastError());
  CU(cudaEventElapsedTime(&ctx->stats.total_ms, ctx->ev0, ctx->ev1));
  const unsigned long long* h = ctx->h_counters;
  ctx->stats.extend_rays = (int64_t)h[CNT_EXTEND_RAYS];
  ctx->stats.shade_lanes = (int64_t)h[CNT_SHADE_LANES];
  ctx->stats.shadow_rays = (int64_t)h[CNT_SHADOW_RAYS];
  ctx->stats.sdf_evals_extend = (int64_t)h[CNT_EVALS_EXTEND];
  ctx->stats.sdf_evals_shadow = (int64_t)h[CNT_EVALS_SHADOW];
  ctx->stats.sdf_evals_normals = (int64_t)h[CNT_EVALS_NORMALS];
  ctx->stats.bulb_iters_extend = (int64_t)h[CNT_BULB_ITERS_EXTEND];
  ctx->stats.bulb_iters_shadow = (int64_t)h[CNT_BULB_ITERS_SHADOW];
  ctx->stats.march_trips_extend = (int64_t)h[CNT_TRIPS_EXTEND];
  ctx->stats.march_trips_shadow = (int64_t)h[CNT_TRIPS_SHADOW];
  {
    int64_t paths = 0;
    for (int idx : ctx->job_tiles) {
      const int tx = idx / ctx->job_nty, ty = idx % ctx->job_nty;
      const int tw = std::min(tx * ctx->job_tw + ctx->job_tw, ctx->job_w) - tx * ctx->job_tw;
      const int th = std::min(ty * ctx->job_th + ctx->job_th, ctx->job_h) - ty * ctx->job_th;
      paths += (int64_t)tw * th * ctx->job_spp;
    }
    ctx->stats.paths = paths;
  }
  for (size_t i = 0; i < ctx->timed_used; ++i) {
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, ctx->timed[i].a, ctx->timed[i].b);
    ctx->stats.kernel_ms[ctx->timed[i].kernel] += ms;
  }
  return RAYN_OK;
}

static int32_t check_planes(RaynContext* ctx, const RaynFilmPlanes* out, bool need_all) {
  if (!out) return fail(ctx, RAYN_ERR_INVALID_ARG, "out is NULL");
  if (!out->color && !out->alpha && !out->background && !out->normal) return fail(ctx, RAYN_ERR_INVALID_ARG, "every film plane is NULL");
  if (need_all && (!out->color || !out->alpha || !out->background || !out->normal))
    return fail(ctx, RAYN_ERR_INVALID_ARG, "a gathered device-space film needs all four planes");
  return RAYN_OK;
}

// ---- NCCL plumbing ---------------------------------------------------------------------------------------
static int32_t nccl_load(RaynContext* ctx) {
  if (g_nccl.handle) return RAYN_OK;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);  // the copy already mapped by the host process (e.g. torch's) wins by soname
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return fail(ctx, RAYN_ERR_NCCL, "cannot load libnccl.so.2: %s", dlerror());
  NcclApi a;
  a.handle = h;
#define SYM(field, name)                                                                     \
  *(void**)(&a.field) = dlsym(h, name);                                                      \
  if (!a.field) return fail(ctx, RAYN_ERR_NCCL, "libnccl.so.2 lacks %s", name);
  SYM(GetUniqueId, "ncclGetUniqueId")
  SYM(CommInitRank, "ncclCommInitRank")
  SYM(CommInitAll, "ncclCommInitAll")
  SYM(CommDestroy, "ncclCommDestroy")
  SYM(AllGather, "ncclAllGather")
  SYM(GroupStart, "ncclGroupStart")
  SYM(GroupEnd, "ncclGroupEnd")
  SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
  g_nccl = a;
  return RAYN_OK;
}

// shard tables + slab storage for a film geometry (uploaded once per geometry, not per frame)
static int32_t comm_prepare(RaynContext* ctx, int W, int H, int tw, int th) {
  RaynComm& c = ctx->comm;
  if (c.W == W && c.H == H && c.tw == tw && c.th == th && c.d_table) return RAYN_OK;
  CU(cudaSetDevice(ctx->device));
  c.shards.clear();
  size_t per = 0;
  for (int r = 0; r < c.world; ++r) {
    c.shards.push_back(shard_of(W, H, tw, th, r, c.world));
    per = std::max(per, c.shards.back().size());
  }
  per = std::max<size_t>(per, 1);
  std::vector<int> table((size_t)c.world * per, -1);
  for (int r = 0; r < c.world; ++r) std::copy(c.shards[r].begin(), c.shards[r].end(), table.begin() + (size_t)r * per);
  CU(cudaStreamSynchronize(ctx->stream));
  cudaFree(c.d_table);
  c.d_table = nullptr;
  CU(cudaMalloc(&c.d_table, table.size() * sizeof(int)));
  CU(cudaMemcpy(c.d_table, table.data(), table.size() * sizeof(int), cudaMemcpyHostToDevice));
  CU(regrow(&c.d_slabs, &c.cap_slabs, (size_t)c.world * per * 10 * tw * th));
  c.W = W, c.H = H, c.tw = tw, c.th = th, c.per_rank = (int)per;
  return RAYN_OK;
}

// pack this rank's tiles into its slab, all-gather in place, ONE unpack kernel over the peers' slabs: all on the render
// stream, zero host synchronisation.  in_group: the caller brackets several contexts with ncclGroupStart/End.
static int32_t gather_pack(RaynContext* ctx, const RaynFilmPlanes* pl) {
  RaynComm& c = ctx->comm;
  int ntx, nty;
  tile_grid_of(c.W, c.H, c.tw, c.th, &ntx, &nty);
  k_film_slab<<<c.per_rank, 256, 0, ctx->stream>>>(c.W, c.H, c.tw, c.th, nty, c.d_table, c.per_rank, c.rank, -1, 0, c.d_slabs, pl->color, pl->alpha,
                                                   pl->background, pl->normal);
  ctx->stats.launches++;
  return RAYN_OK;
}
static int32_t gather_collective(RaynContext* ctx) {
  RaynComm& c = ctx->comm;
  const size_t count = (size_t)c.per_rank * 10 * c.tw * c.th;
  NC(g_nccl.AllGather(c.d_slabs + (size_t)c.rank * count, c.d_slabs, count, kNcclFloat, c.comm, ctx->stream));
  return RAYN_OK;
}
static int32_t gather_unpack(RaynContext* ctx, const RaynFilmPlanes* pl) {
  RaynComm& c = ctx->comm;
  int ntx, nty;
  tile_grid_of(c.W, c.H, c.tw, c.th, &ntx, &nty);
  k_film_slab<<<c.world * c.per_rank, 256, 0, ctx->stream>>>(c.W, c.H, c.tw, c.th, nty, c.d_table, c.per_rank, 0, c.rank, 1, c.d_slabs, pl->color,
                                                             pl->alpha, pl->background, pl->normal);
  ctx->stats.launches++;
  CU(cudaGetLastError());
  return RAYN_OK;
}
static int32_t gather_enqueue(RaynContext* ctx, int W, int H, int tw, int th, const RaynFilmPlanes* pl, bool in_group) {
  (void)in_group;
  if (!ctx->comm.comm) return fail(ctx, RAYN_ERR_INVALID_ARG, "no communicator: call rayn_b200_comm_init_rank / comm_init_all first");
  int32_t rc = comm_prepare(ctx, W, H, tw, th);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  timed_begin(ctx, RAYN_K_GATHER);
  if ((rc = gather_pack(ctx, pl))) return rc;
  if ((rc = gather_collective(ctx))) return rc;
  if ((rc = gather_unpack(ctx, pl))) return rc;
  timed_end(ctx, RAYN_K_GATHER, 0);
  return RAYN_OK;
}

extern "C" {

int32_t rayn_b200_render_frame(RaynContext* ctx, const RaynFrameDesc* f, const RaynFilmPlanes* out) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  int32_t rc = check_planes(ctx, out, false);
  if (rc) return rc;
  if ((rc = render_enqueue(ctx, f, out, nullptr, nullptr))) return rc;
  if ((rc = copy_out_enqueue(ctx, out))) {
    render_finish(ctx);
    return rc;
  }
  return render_finish(ctx);
}

int32_t rayn_b200_sync(RaynContext* ctx) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  return RAYN_OK;
}

// ---- communicator ------------------------------------------------------------------------------------------
int32_t rayn_b200_comm_unique_id(uint8_t* out_id) {
  RaynContext* ctx = nullptr;
  if (!out_id) return fail(nullptr, RAYN_ERR_INVALID_ARG, "out_id is NULL");
  int32_t rc = nccl_load(nullptr);
  if (rc) return rc;
  ncclUniqueId id;
  NC(g_nccl.GetUniqueId(&id));
  memcpy(out_id, id.internal, RAYN_COMM_ID_BYTES);
  return RAYN_OK;
}
int32_t rayn_b200_comm_init_rank(RaynContext* ctx, const uint8_t* id_bytes, int32_t rank, int32_t world) {
  if (!ctx || !id_bytes) return fail(ctx, RAYN_ERR_INVALID_ARG, "comm_init_rank: NULL argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, RAYN_ERR_INVALID_ARG, "comm_init_rank: rank %d of %d", rank, world);
  int32_t rc = nccl_load(ctx);
  if (rc) return rc;
  rayn_b200_comm_destroy(ctx);
  CU(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  memcpy(id.internal, id_bytes, RAYN_COMM_ID_BYTES);
  NC(g_nccl.CommInitRank(&ctx->comm.comm, world, id, rank));
  ctx->comm.rank = rank, ctx->comm.world = world;
  return RAYN_OK;
}
int32_t rayn_b200_comm_init_all(RaynContext* const* ctxs, int32_t n) {
  RaynContext* ctx = (ctxs && n > 0) ? ctxs[0] : nullptr;
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "comm_init_all: no contexts");
  int32_t rc = nccl_load(ctx);
  if (rc) return rc;
  std::vector<int> devs(n);
  std::vector<ncclComm_t> comms(n, nullptr);
  for (int i = 0; i < n; ++i) {
    if (!ctxs[i]) return fail(ctx, RAYN_ERR_INVALID_ARG, "comm_init_all: ctxs[%d] is NULL", i);
    for (int j = 0; j < i; ++j)
      if (ctxs[j]->device == ctxs[i]->device) return fail(ctx, RAYN_ERR_INVALID_ARG, "comm_init_all: device %d used twice", ctxs[i]->device);
    rayn_b200_comm_destroy(ctxs[i]);
    devs[i] = ctxs[i]->device;
  }
  NC(g_nccl.CommInitAll(comms.data(), n, devs.data()));
  for (int i = 0; i < n; ++i) ctxs[i]->comm.comm = comms[i], ctxs[i]->comm.rank = i, ctxs[i]->comm.world = n;
  return RAYN_OK;
}
int32_t rayn_b200_comm_info(const RaynContext* ctx, int32_t* rank, int32_t* world) {
  if (!ctx) return RAYN_ERR_INVALID_ARG;
  if (rank) *rank = ctx->comm.rank;
  if (world) *world = ctx->comm.comm ? ctx->comm.world : 0;
  return RAYN_OK;
}
int32_t rayn_b200_shard_tiles(int32_t W, int32_t H, int32_t tw, int32_t th, int32_t rank, int32_t world, int32_t* out, int32_t cap) {
  if (W <= 0 || H <= 0 || tw <= 0 || th <= 0 || world < 1 || rank < 0 || rank >= world) return -1;
  const std::vector<int> v = shard_of(W, H, tw, th, rank, world);
  if (out && cap >= (int32_t)v.size()) std::copy(v.begin(), v.end(), out);
  return (int32_t)v.size();
}

int32_t rayn_b200_film_gather(RaynContext* ctx, int32_t W, int32_t H, int32_t tw, int32_t th, const RaynFilmPlanes* pl) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  if (W <= 0 || H <= 0 || tw <= 0 || th <= 0) return fail(ctx, RAYN_ERR_INVALID_ARG, "film_gather: bad geometry");
  int32_t rc = check_planes(ctx, pl, true);
  if (rc) return rc;
  if (pl->space != RAYN_MEM_DEVICE) return fail(ctx, RAYN_ERR_INVALID_ARG, "film_gather: planes must be device pointers");
  return gather_enqueue(ctx, W, H, tw, th, pl, false);
}

int32_t rayn_b200_render_frame_sharded(RaynContext* ctx, const RaynFrameDesc* f, const RaynFilmPlanes* out) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  if (!ctx->comm.comm) return fail(ctx, RAYN_ERR_INVALID_ARG, "render_frame_sharded: no communicator on this context");
  if (!f) return fail(ctx, RAYN_ERR_INVALID_ARG, "frame is NULL");
  int32_t rc = check_planes(ctx, out, out && out->space == RAYN_MEM_DEVICE);
  if (rc) return rc;
  const std::vector<int> tiles = shard_of(f->width, f->height, f->tile_w, f->tile_h, ctx->comm.rank, ctx->comm.world);
  RaynFilmPlanes dev;
  if ((rc = render_enqueue(ctx, f, out, &tiles, &dev))) return rc;
  rc = gather_enqueue(ctx, f->width, f->height, f->tile_w, f->tile_h, &dev, false);
  if (!rc) rc = copy_out_enqueue(ctx, out);
  const int32_t rc2 = render_finish(ctx);
  return rc ? rc : rc2;
}

int32_t rayn_b200_render_frame_multi(RaynContext* const* ctxs, int32_t n, const RaynFrameDesc* f, const RaynFilmPlanes* out) {
  RaynContext* ctx = (ctxs && n > 0) ? ctxs[0] : nullptr;
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "render_frame_multi: no contexts");
  if (!f || !out) return fail(ctx, RAYN_ERR_INVALID_ARG, "frame/out is NULL");
  if (f->input_space != RAYN_MEM_HOST || out->space != RAYN_MEM_HOST)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "render_frame_multi: frame inputs and film planes must be host pointers");
  int32_t rc = check_planes(ctx, out, false);
  if (rc) return rc;
  for (int i = 0; i < n; ++i)
    if (!ctxs[i] || !ctxs[i]->comm.comm || ctxs[i]->comm.world != n || ctxs[i]->comm.rank != i)
      return fail(ctx, RAYN_ERR_INVALID_ARG, "render_frame_multi: contexts must come from comm_init_all(ctxs, %d) in the same order", n);
  std::vector<RaynFilmPlanes> dev(n);
  RaynFilmPlanes scratch = *out;  // host-space marker: every context renders into its own device planes
  int32_t first_err = RAYN_OK;
  for (int i = 0; i < n && !first_err; ++i) {
    const std::vector<int> tiles = shard_of(f->width, f->height, f->tile_w, f->tile_h, i, n);
    first_err = render_enqueue(ctxs[i], f, &scratch, &tiles, &dev[i]);
    if (first_err && ctxs[i] != ctx) fail(ctx, first_err, "GPU %d: %s", ctxs[i]->device, ctxs[i]->err.c_str());
  }
  if (!first_err) {
    for (int i = 0; i < n && !first_err; ++i) {
      first_err = comm_prepare(ctxs[i], f->width, f->height, f->tile_w, f->tile_h);
      if (!first_err) {
        cudaSetDevice(ctxs[i]->device);
        first_err = gather_pack(ctxs[i], &dev[i]);
      }
    }
    if (!first_err) {
      g_nccl.GroupStart();
      for (int i = 0; i < n && !first_err; ++i) {
        cudaSetDevice(ctxs[i]->device);
        first_err = gather_collective(ctxs[i]);
      }
      const int gr = g_nccl.GroupEnd();
      if (!first_err && gr) first_err = fail(ctx, RAYN_ERR_NCCL, "ncclGroupEnd: %s", g_nccl.GetErrorString(gr));
    }
    for (int i = 0; i < n && !first_err; ++i) {
      cudaSetDevice(ctxs[i]->device);
      first_err = gather_unpack(ctxs[i], &dev[i]);
    }
    if (!first_err) first_err = copy_out_enqueue(ctx, out);
  }
  for (int i = 0; i < n; ++i) {
    const int32_t rc2 = render_finish(ctxs[i]);
    if (!first_err && rc2) first_err = rc2;
  }
  return first_err;
}

// ---- explicit slab helpers --------------------------------------------------------------------------------------
int64_t rayn_b200_film_slab_floats(int32_t tw, int32_t th, int32_t n_tiles) {
  if (tw <= 0 || th <= 0 || n_tiles < 0) return -1;
  return (int64_t)n_tiles * 10 * tw * th;
}
static int32_t pack_unpack(RaynContext* ctx, int W, int H, int tw, int th, const int32_t* tile_list, int n, const RaynFilmPlanes* pl,
                           float* slab, int unpack) {
  if (!ctx || !pl || !slab || n < 0 || (n && !tile_list) || W <= 0 || H <= 0 || tw <= 0 || th <= 0)
    return fail(ctx, RAYN_ERR_INVALID_ARG, "film pack/unpack: bad argument");
  if (n == 0) return RAYN_OK;
  CU(cudaSetDevice(ctx->device));
  int ntx, nty;
  tile_grid_of(W, H, tw, th, &ntx, &nty);
  for (int i = 0; i < n; ++i)
    if (tile_list[i] < 0 || tile_list[i] >= ntx * nty) return fail(ctx, RAYN_ERR_INVALID_ARG, "film pack/unpack: tile %d out of range", tile_list[i]);
  CU(regrow(&ctx->d_pack_ids, &ctx->cap_pack_ids, (size_t)n));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpyAsync(ctx->d_pack_ids, tile_list, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  k_film_slab<<<n, 256, 0, ctx->stream>>>(W, H, tw, th, nty, ctx->d_pack_ids, n, 0, -1, unpack, slab, pl->color, pl->alpha, pl->background, pl->normal);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(ctx->stream));
  return RAYN_OK;
}
int32_t rayn_b200_film_pack_tiles(RaynContext* ctx, int32_t W, int32_t H, int32_t tw, int32_t th, const int32_t* tile_list, int32_t n_tiles,
                                  const RaynFilmPlanes* planes_dev, float* slab_dev) {
  return pack_unpack(ctx, W, H, tw, th, tile_list, n_tiles, planes_dev, slab_dev, 0);
}
int32_t rayn_b200_film_unpack_tiles(RaynContext* ctx, int32_t W, int32_t H, int32_t tw, int32_t th, const int32_t* tile_list, int32_t n_tiles,
                                    const float* slab_dev, const RaynFilmPlanes* planes_dev) {
  return pack_unpack(ctx, W, H, tw, th, tile_list, n_tiles, planes_dev, const_cast<float*>(slab_dev), 1);
}

// ---- film post-process (film.rs:205-377 arithmetic) -------------------------------------------------
int32_t rayn_b200_film_postprocess(RaynContext* ctx, int32_t mode, int32_t W, int32_t H, const RaynFilmPlanes* pl, uint8_t* out,
                                   int32_t out_space) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  if (mode < 0 || mode > RAYN_POST_ALPHA || W <= 0 || H <= 0 || !pl || !out) return fail(ctx, RAYN_ERR_INVALID_ARG, "film_postprocess: bad argument");
  const bool need_color = mode <= RAYN_POST_COLOR_ONLY, need_bg = mode == RAYN_POST_COLOR_PLUS_BACKGROUND || mode == RAYN_POST_BACKGROUND;
  const bool need_alpha = mode == RAYN_POST_COLOR_ALPHA || mode == RAYN_POST_ALPHA, need_normal = mode == RAYN_POST_WORLD_NORMAL;
  if ((need_color && !pl->color) || (need_bg && !pl->background) || (need_alpha && !pl->alpha) || (need_normal && !pl->normal))
    return fail(ctx, RAYN_ERR_INVALID_ARG, "Attempted to write a channel with insufficient channels");  // film.rs:294-298
  CU(cudaSetDevice(ctx->device));
  const size_t npx = (size_t)W * H, nbytes = npx * post_bytes_per_pixel(mode);
  cudaStream_t st = ctx->stream;
  const float *c = pl->color, *a = pl->alpha, *b = pl->background, *n = pl->normal;
  CU(cudaDeviceSynchronize());
  if (pl->space == RAYN_MEM_HOST) {
    CU(regrow(&ctx->d_planes, &ctx->cap_planes, npx * 10));
    float* d = ctx->d_planes;
    if (need_color) CU(cudaMemcpyAsync(d, pl->color, npx * 12, cudaMemcpyHostToDevice, st));
    if (need_alpha) CU(cudaMemcpyAsync(d + 3 * npx, pl->alpha, npx * 4, cudaMemcpyHostToDevice, st));
    if (need_bg) CU(cudaMemcpyAsync(d + 4 * npx, pl->background, npx * 12, cudaMemcpyHostToDevice, st));
    if (need_normal) CU(cudaMemcpyAsync(d + 7 * npx, pl->normal, npx * 12, cudaMemcpyHostToDevice, st));
    c = d, a = d + 3 * npx, b = d + 4 * npx, n = d + 7 * npx;
  }
  unsigned char* dout = out;
  if (out_space == RAYN_MEM_HOST) {
    CU(regrow(&ctx->d_post, &ctx->cap_post, nbytes));
    dout = ctx->d_post;
  }
  k_postprocess<<<(unsigned)((npx + 255) / 256), 256, 0, st>>>(mode, W, H, c, a, b, n, dout);
  CU(cudaGetLastError());
  if (out_space == RAYN_MEM_HOST) CU(cudaMemcpyAsync(out, dout, nbytes, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return RAYN_OK;
}

int32_t rayn_b200_device_frame_inputs(RaynContext* ctx, int32_t W, int32_t H, int32_t spp, int32_t sets_1d, int32_t sets_2d, uint64_t offset,
                                      float* s1, float* s2, float* scramble) {
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");
  if (spp <= 0 || sets_1d < 0 || sets_2d < 0 || (sets_1d && !s1) || (sets_2d && !s2) || (scramble && (W <= 0 || H <= 0)))
    return fail(ctx, RAYN_ERR_INVALID_ARG, "device_frame_inputs: bad argument");
  CU(cudaSetDevice(ctx->device));
  CU(cudaDeviceSynchronize());
  const long long n = (long long)spp * (sets_1d + sets_2d);
  if (n > 0) k_gen_rd_tables<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(spp, sets_1d, sets_2d, offset, s1, s2);
  if (scramble) k_gen_scramble<<<(unsigned)(((long long)W * H + 255) / 256), 256, 0, ctx->stream>>>(W, H, scramble);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(ctx->stream));
  return RAYN_OK;
}

// ---- known-answer entry points ----------------------------------------------------------------------
#define KAT_PROLOGUE                                                     \
  if (!ctx) return fail(nullptr, RAYN_ERR_INVALID_ARG, "ctx is NULL");   \
  if (n < 0) return fail(ctx, RAYN_ERR_INVALID_ARG, "n < 0");            \
  CU(cudaSetDevice(ctx->device));                                        \
  if (n == 0) return RAYN_OK;                                            \
  DevTmp tmp;                                                            \
  cudaError_t e = cudaSuccess;                                           \
  const unsigned blocks = (unsigned)((n + 127) / 128);
#define KAT_EPILOGUE(dst, src, count, T)                                              \
  CU(e);                                                                              \
  CU(cudaGetLastError());                                                             \
  CU(cudaStreamSynchronize(ctx->stream));                                             \
  CU(cudaMemcpy(dst, src, (size_t)(count) * sizeof(T), cudaMemcpyDeviceToHost));

int32_t rayn_b200_kat_detmath(RaynContext* ctx, int32_t op, int64_t n, const float* a, const float* b, float* out) {
  KAT_PROLOGUE
  if (op < 0 || op > 7 || !a || !out) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_detmath: bad argument");
  float* da = tmp.up(a, n, &e);
  float* db = tmp.up(b ? b : a, n, &e);
  float* dout = tmp.up<float>(nullptr, n, &e);
  CU(e);
  k_kat_detmath<<<blocks, 128, 0, ctx->stream>>>(op, n, da, db, dout);
  KAT_EPILOGUE(out, dout, n, float)
  return RAYN_OK;
}
int32_t rayn_b200_kat_sdf_dist(RaynContext* ctx, const RaynHitable* sdf, int64_t n, const float* points3, float* out) {
  KAT_PROLOGUE
  if (!sdf || !points3 || !out) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_sdf_dist: NULL");
  float* dp = tmp.up(points3, 3 * n, &e);
  float* dout = tmp.up<float>(nullptr, n, &e);
  CU(e);
  k_kat_sdf_dist<<<blocks, 128, 0, ctx->stream>>>(*sdf, n, dp, dout);
  KAT_EPILOGUE(out, dout, n, float)
  return RAYN_OK;
}
int32_t rayn_b200_kat_sdf_dist2(RaynContext* ctx, const RaynHitable* sdf, int32_t variant, int64_t n, const float* points3, float* out) {
  KAT_PROLOGUE
  if (!sdf || !points3 || !out) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_sdf_dist2: NULL");
  if (sdf->kind == RAYN_HITABLE_SPHERE) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_sdf_dist2: not an SDF");
  int v = variant < 0 ? sdf_variant(*sdf, div3_verified(ctx, *sdf)) : variant;
  const bool v_fast = v == SDFV_BOX_12_FAST || v == SDFV_BOX_N_FAST, v_div3 = v == SDFV_BOX_12_DIV3 || v == SDFV_BOX_N_DIV3;
  if (v >= SDFV_COUNT || (v == SDFV_BULB) != (sdf->kind == RAYN_HITABLE_MANDELBULB) || ((v_fast || v_div3) && !sdf_box_fast_ok(*sdf)) ||
      ((v == SDFV_BOX_12_FAST || v == SDFV_BOX_12_DIV3) && sdf->iterations != 12) || (v_div3 && !div3_verified(ctx, *sdf)))
    return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_sdf_dist2: variant %d does not fit the hitable", v);
  float* dp = tmp.up(points3, 3 * n, &e);
  float* dout = tmp.up<float>(nullptr, n, &e);
  CU(e);
  DISPATCH_SDFV(v, (k_kat_sdf_dist2<V><<<(unsigned)((n / 2 + 128) / 128), 128, 0, ctx->stream>>>(*sdf, 1.0f, n, dp, dout)));
  KAT_EPILOGUE(out, dout, n, float)
  return RAYN_OK;
}
int32_t rayn_b200_kat_fastdiv(RaynContext* ctx, float num, uint32_t first_bits, int64_t n, int64_t* out_mismatches) {
  if (!ctx || !out_mismatches || n < 0) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_fastdiv: bad argument");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemsetAsync(ctx->d_kat, 0, sizeof(unsigned long long), ctx->stream));
  if (n > 0) k_kat_fastdiv<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(num, first_bits, n, ctx->d_kat);
  CU(cudaGetLastError());
  unsigned long long h = 0;
  CU(cudaMemcpyAsync(&h, ctx->d_kat, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  *out_mismatches = (int64_t)h;
  return RAYN_OK;
}
int32_t rayn_b200_kat_sdf_hit(RaynContext* ctx, const RaynHitable* sdf, const RaynRenderConsts* consts, int64_t n, const float* origins3,
                              const float* dirs3, const float* t_max, float thr_scale, int32_t thr_const, float* out_t) {
  KAT_PROLOGUE
  if (!sdf || !consts || !origins3 || !dirs3 || !t_max || !out_t) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_sdf_hit: NULL");
  float* dor = tmp.up(origins3, 3 * n, &e);
  float* ddi = tmp.up(dirs3, 3 * n, &e);
  float* dtm = tmp.up(t_max, n, &e);
  float* dout = tmp.up<float>(nullptr, n, &e);
  CU(e);
  Thr thr;
  thr.scale = thr_scale;
  thr.is_const = thr_const;
  k_kat_sdf_hit<<<blocks, 128, 0, ctx->stream>>>(*sdf, *consts, n, dor, ddi, dtm, thr, dout);
  KAT_EPILOGUE(out_t, dout, n, float)
  return RAYN_OK;
}
int32_t rayn_b200_kat_occluded(RaynContext* ctx, int64_t n, const float* start3, const float* end3, float* out) {
  KAT_PROLOGUE
  if (!ctx->has_scene) return fail(ctx, RAYN_ERR_NO_SCENE, "kat_occluded before upload_scene");
  if (!start3 || !end3 || !out) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_occluded: NULL");
  float* ds = tmp.up(start3, 3 * n, &e);
  float* de = tmp.up(end3, 3 * n, &e);
  float* dout = tmp.up<float>(nullptr, n, &e);
  CU(e);
  if (ctx->tables)
    k_kat_occluded<<<blocks, 128, 0, ctx->stream>>>(ctx->tscene, n, ds, de, dout);
  else
    k_kat_occluded<<<blocks, 128, 0, ctx->stream>>>(ctx->scene, n, ds, de, dout);
  KAT_EPILOGUE(out, dout, n, float)
  return RAYN_OK;
}
int32_t rayn_b200_kat_closest_hit(RaynContext* ctx, int32_t depth, int64_t n, const float* origins3, const float* dirs3, float* out_t,
                                  int32_t* out_obj) {
  KAT_PROLOGUE
  if (!ctx->has_scene) return fail(ctx, RAYN_ERR_NO_SCENE, "kat_closest_hit before upload_scene");
  if (!origins3 || !dirs3 || !out_t || !out_obj) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_closest_hit: NULL");
  float* dor = tmp.up(origins3, 3 * n, &e);
  float* ddi = tmp.up(dirs3, 3 * n, &e);
  float* dt = tmp.up<float>(nullptr, n, &e);
  int* dobj = tmp.up<int>(nullptr, n, &e);
  CU(e);
  if (ctx->tables)
    k_kat_closest_hit<<<blocks, 128, 0, ctx->stream>>>(ctx->tscene, make_thr(ctx->scene.cam, depth), n, dor, ddi, dt, dobj);
  else
    k_kat_closest_hit<<<blocks, 128, 0, ctx->stream>>>(ctx->scene, make_thr(ctx->scene.cam, depth), n, dor, ddi, dt, dobj);
  KAT_EPILOGUE(out_t, dt, n, float)
  CU(cudaMemcpy(out_obj, dobj, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost));
  return RAYN_OK;
}

int32_t rayn_b200_kat_light_sample(RaynContext* ctx, const RaynLight* light, int64_t n, const float* s0, const float* s1, const float* points3,
                                   float* out_point3, float* out_pdf) {
  KAT_PROLOGUE
  if (!light || !s0 || !s1 || !points3 || !out_point3 || !out_pdf) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_light_sample: NULL");
  float *d0 = tmp.up(s0, n, &e), *d1 = tmp.up(s1, n, &e), *dp = tmp.up(points3, 3 * n, &e);
  float *dpt = tmp.up<float>(nullptr, 3 * n, &e), *dpdf = tmp.up<float>(nullptr, n, &e);
  CU(e);
  k_kat_light_sample<<<blocks, 128, 0, ctx->stream>>>(*light, n, d0, d1, dp, dpt, dpdf);
  KAT_EPILOGUE(out_point3, dpt, 3 * n, float)
  CU(cudaMemcpy(out_pdf, dpdf, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  return RAYN_OK;
}
int32_t rayn_b200_kat_light_sample_volume(RaynContext* ctx, const RaynLight* light, int64_t n, const float* sample, const float* origins3,
                                          const float* dirs3, const float* t_max, float* out_t, float* out_pdf) {
  KAT_PROLOGUE
  if (!light || !sample || !origins3 || !dirs3 || !t_max || !out_t || !out_pdf) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_light_sample_volume: NULL");
  float *ds = tmp.up(sample, n, &e), *dor = tmp.up(origins3, 3 * n, &e), *ddi = tmp.up(dirs3, 3 * n, &e), *dtm = tmp.up(t_max, n, &e);
  float *dt = tmp.up<float>(nullptr, n, &e), *dpdf = tmp.up<float>(nullptr, n, &e);
  CU(e);
  k_kat_light_sample_volume<<<blocks, 128, 0, ctx->stream>>>(*light, n, ds, dor, ddi, dtm, dt, dpdf);
  KAT_EPILOGUE(out_t, dt, n, float)
  CU(cudaMemcpy(out_pdf, dpdf, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  return RAYN_OK;
}
int32_t rayn_b200_kat_bsdf(RaynContext* ctx, const RaynMaterial* mat, int64_t n, const float* normals3, const float* wo3, const float* s1d,
                           const float* u4, float* out_wi3, float* out_f3, float* out_pdf, float* out_feval3) {
  KAT_PROLOGUE
  if (!mat || !normals3 || !wo3 || !s1d || !u4 || !out_wi3 || !out_f3 || !out_pdf || !out_feval3) return fail(ctx, RAYN_ERR_INVALID_ARG, "kat_bsdf: NULL");
  float *dn = tmp.up(normals3, 3 * n, &e), *dw = tmp.up(wo3, 3 * n, &e), *ds = tmp.up(s1d, n, &e), *du = tmp.up(u4, 4 * n, &e);
  float *dwi = tmp.up<float>(nullptr, 3 * n, &e), *df = tmp.up<float>(nullptr, 3 * n, &e), *dpdf = tmp.up<float>(nullptr, n, &e),
        *dfe = tmp.up<float>(nullptr, 3 * n, &e);
  CU(e);
  k_kat_bsdf<<<blocks, 128, 0, ctx->stream>>>(*mat, n, dn, dw, ds, du, dwi, df, dpdf, dfe);
  KAT_EPILOGUE(out_wi3, dwi, 3 * n, float)
  CU(cudaMemcpy(out_f3, df, (size_t)3 * n * sizeof(float), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(out_pdf, dpdf, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(out_feval3, dfe, (size_t)3 * n * sizeof(float), cudaMemcpyDeviceToHost));
  return RAYN_OK;
}

}  // extern "C"
