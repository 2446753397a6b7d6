/*
 * rayn_b200.h — C ABI of the B200-native wavefront path tracer that replaces the
 * render hot path of fu5ha/rayn (reference @ 6486a86).
 *
 * The ONE reference call this boundary replaces is
 *     Film::render_frame_into(world, camera, integrator, filter, tile_size,
 *                             frame, time_range, samples)
 * (reference src/film.rs:382-395, called once per frame from src/main.rs:64-73).
 *
 * The reference has no FFI: its extension surface is Rust traits with `dyn` objects
 * (src/hitable.rs:8-18, src/material.rs:11-38, src/light.rs:5-17, src/camera.rs:5-19).
 * Trait objects cannot cross to a GPU, so every trait implementor the reference ships
 * becomes a tagged plain-old-data descriptor here.  Insertion ORDER of hitables,
 * materials and lights is semantic (closest-hit fold order src/hitable.rs:177-198,
 * bin order src/hitable.rs:116-133) and is preserved.
 *
 * Everything is plain C: fixed-width ints, floats, pointers and sizes.  No exception
 * ever unwinds across this boundary; every call returns a status code
 * (the reference panics / unwraps instead: src/main.rs:32,45,96, src/film.rs:127,667).
 *
 * A Rust `extern "C"` block for this header is mechanical; INTEGRATION.md shows it.
 */
#ifndef RAYN_B200_H
#define RAYN_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RAYN_B200_ABI_VERSION 2

/* ---- limits -----------------------------------------------------------------------
 * The reference's stores are unbounded `Vec<Box<dyn ..>>` (src/hitable.rs:143, src/material.rs:58, src/world.rs:7-13).
 * A scene of at most 16 hitables, 16 materials and 16 lights rides in the kernel-parameter constant bank (warp-uniform
 * operands then cost no load; setup.rs needs 7 / 4 / 5); a larger one is uploaded once into tables in device memory that
 * the context owns.  Both render the same film.  upload_scene returns RAYN_ERR_INVALID_ARG, naming the limit, beyond:
 *   RAYN_MAX_HITABLES / RAYN_MAX_MATERIALS: the per-tile bin tables hold one row entry per hitable;
 *   RAYN_MAX_LIGHTS: CONTRACT CHANGE vs the reference - the shading kernels exchange a packet's light choices one byte each;
 *   RAYN_MAX_SDF_HITABLES: CONTRACT CHANGE vs the reference - every SDF hitable costs its own march, normals and shadow
 *     kernel per depth and its own shadow-segment queue (pass memory per path grows with the SDF count).              */
#define RAYN_MAX_HITABLES 1024
#define RAYN_MAX_MATERIALS 1024
#define RAYN_MAX_LIGHTS 256
#define RAYN_MAX_SDF_HITABLES 16
#define RAYN_FIS_TABLE_SIZE 512 /* FILTER_TABLE_SIZE, src/filter.rs:187 */

/* ---- status codes ---------------------------------------------------------------- */
typedef enum RaynStatus {
  RAYN_OK = 0,
  RAYN_ERR_INVALID_ARG = 1,
  RAYN_ERR_UNSUPPORTED = 2, /* representable in rayn, not in this build (e.g. vm != 2)   */
  RAYN_ERR_CUDA = 3,
  RAYN_ERR_OOM = 4,
  RAYN_ERR_NO_SCENE = 5,
  RAYN_ERR_NO_DEVICE = 6,
  RAYN_ERR_NCCL = 7      /* NCCL missing (dlopen) or a collective failed                    */
} RaynStatus;

/* ---- Hitable (src/hitable.rs:8-18) ------------------------------------------------ */
typedef enum RaynHitableKind {
  RAYN_HITABLE_SPHERE = 0,     /* Sphere<TR>, src/sphere.rs:7-21 (constant centre)          */
  RAYN_HITABLE_MANDELBOX = 1,  /* TracedSDF<MandelBox>, src/sdf.rs:12-23,104-141            */
  RAYN_HITABLE_MANDELBULB = 2  /* TracedSDF<Mandelbulb>: AUTHORED here, not in the reference */
} RaynHitableKind;

typedef struct RaynHitable {
  int32_t kind;     /* RaynHitableKind                                                     */
  int32_t material; /* MaterialHandle, index into materials[] (src/material.rs:55-56)      */
  /* Sphere::new(centre, radius, material), src/sphere.rs:14-20                            */
  float center[3];
  float radius;
  /* MandelBox::new(iterations, BoxFold::new(l), SphereFold::new(min_r, fixed_r), scale),
   * src/sdf.rs:113-123,150-158,171-179.  The two radii are stored SQUARED, computed by the
   * host in f32 exactly as SphereFold::new does (src/sdf.rs:173-174).                     */
  int32_t iterations;
  float box_l;
  float min_rad_sq;
  float fixed_rad_sq;
  float scale;
  /* Mandelbulb (authored): power is fixed to 8 in this build; bailout radius.             */
  int32_t bulb_power;
  float bulb_bailout;
  /* Sphere<TR> with a time-varying centre (SURVEY §8f rank 4): centre(t) = center + center_velocity * t,
   * i.e. what the closure `|t| center + velocity * t` gives through `impl WSequenced<Wec3> for Fn(f32)->Vec3`
   * (src/animation.rs:62-67) - which evaluates the closure at LANE 0's time for the whole 4-lane packet.
   * All-zero velocity = the constant `impl_inherent_wsequenced` path (animation.rs:52).               */
  float center_velocity[3];
} RaynHitable;

/* ---- Material / BSDF (src/material.rs:11-38) -------------------------------------- */
typedef enum RaynMaterialKind {
  RAYN_MATERIAL_LAMBERTIAN = 0, /* src/material.rs:86-142                                   */
  RAYN_MATERIAL_DIELECTRIC = 1, /* src/material.rs:144-257; roughness = REMAPPED exponent   */
  RAYN_MATERIAL_SKY = 2,        /* src/material.rs:394-449                                  */
  RAYN_MATERIAL_EMISSIVE = 3    /* src/material.rs:451-520                                  */
} RaynMaterialKind;

typedef struct RaynMaterial {
  int32_t kind;
  float albedo[3];     /* Lambertian / Dielectric                                          */
  float roughness;     /* Dielectric: the Phong exponent AFTER new_remap (material.rs:167-174) */
  float sky_top[3];    /* Sky::new(top, bottom)                                            */
  float sky_bottom[3];
  float emission[3];   /* Emissive::new_splat                                              */
} RaynMaterial;

/* ---- Light (src/light.rs:5-17): SphereLight::new(pos, rad, emission) :27-34 -------- */
typedef struct RaynLight {
  float pos[3];
  float rad;
  float emission[3];
} RaynLight;

/* ---- Camera (src/camera.rs:5-19) --------------------------------------------------- */
typedef enum RaynCameraKind {
  RAYN_CAMERA_PINHOLE = 0,     /* src/camera.rs:42-119  */
  RAYN_CAMERA_THINLENS = 1,    /* src/camera.rs:121-213 */
  RAYN_CAMERA_ORTHOGRAPHIC = 2 /* src/camera.rs:215-285 */
} RaynCameraKind;

/* The derived fields are what the reference constructors store (camera.rs:52-72,
 * 133-157,227-241); the HOST computes them (tan etc. are host-side f32 libm there too),
 * so they are inputs on both sides of a parity comparison.                               */
typedef struct RaynCamera {
  int32_t kind;
  float half_size[2];    /* (half_width, half_height)                                      */
  float full_size[2];    /* orthographic only                                              */
  float half_pixel_size; /* half_height / res.y, or pixel_size / 2 for orthographic        */
  float origin[3];
  float at[3];
  float up[3];
  float focus[3];        /* thin lens: focus point                                         */
  float aperture;        /* thin lens                                                      */
  /* linear-in-time camera parameters, same closure semantics as RaynHitable.center_velocity
   * (camera.rs:90-92,177-182,258-260 sample origin/at/up/focus at the packet's time): a closure-backed
   * WSequenced<Wec3> is evaluated at LANE 0's time (animation.rs:62-67).                                  */
  float origin_velocity[3];
  float at_velocity[3];
  float up_velocity[3];
  float focus_velocity[3];
  /* EXTENSION, no reference counterpart: aperture(t) = aperture + aperture_rate * t0 (lane-0 time).  The reference
   * implements closure-backed WSequenced only for Fn(f32)->Vec3; an f32 parameter can only be a constant there
   * (impl_wsequenced_for_sequenced, animation.rs:51-53).  Keep 0 for reference behaviour.                       */
  float aperture_rate;
} RaynCamera;

/* ---- VolumeParams (src/volume.rs:2-5): Option<f32> pairs --------------------------- */
typedef struct RaynVolume {
  int32_t has_scattering;
  float coeff_scattering;
  int32_t has_extinction;
  float coeff_extinction;
} RaynVolume;

/* ---- compile-time constants of the reference that leak into the hot path ----------- */
typedef struct RaynRenderConsts {
  float world_radius;      /* WORLD_RADIUS, src/setup.rs:33 (t_max = 2x, film.rs:556)      */
  float sdf_detail_scale;  /* SDF_DETAIL_SCALE, src/setup.rs:37                            */
  int32_t max_marches;     /* MAX_MARCHES = 256, src/sdf.rs:9                              */
  int32_t max_vis_marches; /* MAX_VIS_MARCHES = 100, src/sdf.rs:10                         */
} RaynRenderConsts;

/* ---- World (src/world.rs:7-13) + the selected camera ------------------------------- */
typedef struct RaynSceneDesc {
  int32_t n_hitables;
  const RaynHitable* hitables;
  int32_t n_materials;
  const RaynMaterial* materials;
  int32_t n_lights;
  const RaynLight* lights;
  RaynCamera camera;
  RaynVolume volume;
  RaynRenderConsts consts;
} RaynSceneDesc;

typedef enum RaynMemSpace { RAYN_MEM_HOST = 0, RAYN_MEM_DEVICE = 1 } RaynMemSpace;

/* ---- one call of render_frame_into (src/film.rs:382-395) --------------------------- */
typedef struct RaynFrameDesc {
  int32_t width, height;   /* Film.res                                                     */
  int32_t tile_w, tile_h;  /* tile_size; main.rs passes 16x16                              */
  int32_t samples;         /* SAMPLES; spp = 4*samples (film.rs:439,463-464)               */
  int32_t max_bounces;     /* PathTracingIntegrator.max_bounces (integrator.rs:33-36)      */
  int32_t volume_marches;  /* must be 2: samples_1d[3],[4] are hard-wired (integrator.rs:138,175) */
  int32_t frame;           /* only labels the sample tables here                           */
  float t0, t1;            /* time_range (film.rs:390,454,509-512)                         */
  /* Host-owned sampler state (src/sampler.rs:11-15), passed so seeds match by construction */
  int32_t sets_1d;         /* >= 1 + (mb+1)*(3+vm)   (film.rs:431, integrator.rs:39-41)    */
  int32_t sets_2d;         /* >= 2 + (mb+1)*(12+8vm) (film.rs:432, integrator.rs:43-45)    */
  const float* samples_1d; /* [spp * sets_1d]                                              */
  const float* samples_2d; /* [2 * spp * sets_2d]                                          */
  const float* scramble;   /* [width*height], per-pixel Cranley-Patterson shift (film.rs:460-461) */
  const float* fis_inverse_cdf; /* [512], FilterImportanceSampler (filter.rs:189-218)      */
  int32_t input_space;     /* RaynMemSpace of the four pointers above                      */
  /* multi-GPU sharding: this call renders tiles with (tile_index % tile_stride) == tile_offset,
   * tile_index = tile_x * n_tiles_y + tile_y (film.rs:401-425).  1-GPU: stride 1, offset 0. */
  int32_t tile_offset;
  int32_t tile_stride;
  /* optional explicit shard: if tile_list != NULL (HOST pointer, n_tile_list entries, each a
   * tile_index, ascending) it replaces offset/stride.  Lets the host pick any interleave,
   * e.g. the diagonal (tile_x + tile_y) % N that balances centre-weighted fractal scenes.      */
  const int32_t* tile_list;
  int32_t n_tile_list;
} RaynFrameDesc;

/* ---- Film channel planes (src/film.rs:103-120), row-major, y up, already / spp ------
 * Any plane pointer may be NULL: that channel is not written, like a Film<N> created without it
 * (film.rs:175-203; add_sample ignores absent channels, film.rs:167-172).                  */
typedef struct RaynFilmPlanes {
  float* color;      /* [3*W*H] Srgb                                                       */
  float* alpha;      /* [W*H]                                                              */
  float* background; /* [3*W*H]                                                            */
  float* normal;     /* [3*W*H] WorldNormal                                                */
  int32_t space;     /* RaynMemSpace                                                       */
} RaynFilmPlanes;

typedef struct RaynConfig {
  int32_t device;            /* CUDA device ordinal                                        */
  int64_t max_paths_per_pass;/* queue capacity in paths; 0 = default                       */
  int32_t flags;             /* RAYN_FLAG_*                                                */
} RaynConfig;

#define RAYN_FLAG_TIMING 1       /* record per-kernel CUDA-event times into RaynStats      */
#define RAYN_FLAG_SIMPLE_MARCH 2 /* TEST BUILD ONLY (-DRAYN_LEGACY_KERNELS, librayn_b200_legacy.so): round-1 v0
                                    one-thread-per-ray kernels; RAYN_ERR_UNSUPPORTED in the product library */

#define RAYN_FLAG_NO_FOLD_ALL 64 /* keep the closest-hit fold in insertion order even for [spheres] Mandelbox [spheres] scenes  */
#define RAYN_FLAG_NO_DIV3 32     /* never select the three-operation sphere-fold division (see rayn_b200_debug_sdf_variant) */
#define RAYN_FLAG_NO_GRAPH 16    /* launch every kernel directly; by default small single-pass frames (launch bound) are
                                    captured once into a CUDA graph and replayed with one launch                */
#define RAYN_FLAG_SCENE_TABLES 4 /* upload every scene into device-memory tables, also one that fits the parameter block
                                    (test and measurement hook: the film is the same either way)                  */

#define RAYN_STAT_KERNELS 12
typedef struct RaynStats {
  int64_t launches;                 /* kernels launched by the last render call            */
  int64_t passes;                   /* tile passes                                         */
  int64_t paths;                    /* camera paths generated = samples rendered           */
  int64_t extend_rays;              /* rays through K2 (closest hit), all depths           */
  int64_t shade_lanes;              /* valid lanes shaded, all depths                      */
  int64_t shadow_rays;              /* shadow segments tested (K5)                         */
  int64_t sdf_evals_extend;         /* SDF dist() evaluations inside K2                    */
  int64_t sdf_evals_shadow;         /* SDF dist() evaluations inside K5                    */
  float kernel_ms[RAYN_STAT_KERNELS];   /* RAYN_FLAG_TIMING: summed device ms per kernel   */
  int64_t kernel_launches[RAYN_STAT_KERNELS];
  float total_ms;                   /* device ms of the last render call (events)          */
  int64_t sdf_evals_normals;        /* SDF dist() evaluations of get_shading_info (4 per SDF shading lane) */
  int64_t bulb_iters_extend;        /* Mandelbulb iterations actually run inside K2 (data dependent)       */
  int64_t bulb_iters_shadow;        /* ... inside K5                                                       */
  int64_t reserved_;                /* 1 when the last frame ran as ONE CUDA-graph launch (captured or replayed) */
  int64_t march_trips_extend;       /* warp-level distance-evaluation trips of K2: sdf_evals_extend / (64 * trips) = busy march slots */
  int64_t march_trips_shadow;       /* ... of K5                                                                                      */
} RaynStats;

/* indices into kernel_ms / kernel_launches */
enum {
  RAYN_K_RAYGEN = 0,
  RAYN_K_EXTEND = 1,
  RAYN_K_BIN = 2,
  RAYN_K_SHADE_PRE = 3,
  RAYN_K_SHADOW = 4,
  RAYN_K_SHADE_POST = 5,
  RAYN_K_COMPACT = 6,
  RAYN_K_RESOLVE = 7,
  RAYN_K_MISC = 8,
  RAYN_K_NORMALS = 9,
  RAYN_K_EXTEND_SPHERES = 10,
  RAYN_K_GATHER = 11
};

typedef struct RaynContext RaynContext;

/* ---- lifecycle --------------------------------------------------------------------- */
int32_t rayn_b200_abi_version(void);
/* 1 if this library was built with `wide` f32x4::mul_add FUSED (rayn built with -C target-feature=+fma), 0 for the
 * default: unfused, what a stock `cargo run --release` of the reference produces (oracle/README.md A6).          */
int32_t rayn_b200_muladd_fused(void);
int32_t rayn_b200_create(const RaynConfig* cfg, RaynContext** out_ctx);
void rayn_b200_destroy(RaynContext* ctx);
const char* rayn_b200_last_error(const RaynContext* ctx); /* ctx may be NULL: global slot */

/* World -> device.  Replaces the `&world` argument of film.rs:384.                      */
int32_t rayn_b200_upload_scene(RaynContext* ctx, const RaynSceneDesc* scene);

/* The drop-in for Film::render_frame_into (film.rs:382-628) + tile_finished (:660-691).
 * Host pointers: inputs are copied H2D and planes D2H inside the call.
 * Device pointers: nothing is copied; planes are written in place on the device.        */
int32_t rayn_b200_render_frame(RaynContext* ctx, const RaynFrameDesc* frame,
                               const RaynFilmPlanes* out);

int32_t rayn_b200_get_stats(const RaynContext* ctx, RaynStats* out);

/* ---- multi-GPU: film tiles shard across GPUs, NCCL only for the final film gather -------------------------
 * The reference's only parallelism is one rayon task per tile over shared read-only state (film.rs:640-649); the
 * multi-GPU form of that is one context per GPU, each rendering the tiles `(tile_x + tile_y) % world == rank`
 * (interleaved: fractal scenes are centre-weighted), and ONE all-gather of dense tile slabs at the end of the frame.
 * The context owns the NCCL communicator (SURVEY §8b "Threading"):
 *   one process per GPU : rank 0 calls comm_unique_id, the host distributes the 128 bytes by any means, every rank
 *                         calls comm_init_rank on its context;
 *   one process, n GPUs : comm_init_all(ctxs, n)  (ncclCommInitAll), then render_frame_multi.
 * NCCL is dlopen()ed ("libnccl.so.2") at the first comm call: the library has no link-time NCCL dependency.      */
#define RAYN_COMM_ID_BYTES 128
int32_t rayn_b200_comm_unique_id(uint8_t out_id[RAYN_COMM_ID_BYTES]);
int32_t rayn_b200_comm_init_rank(RaynContext* ctx, const uint8_t id[RAYN_COMM_ID_BYTES], int32_t rank, int32_t world);
int32_t rayn_b200_comm_init_all(RaynContext* const* ctxs, int32_t n);
int32_t rayn_b200_comm_destroy(RaynContext* ctx);
int32_t rayn_b200_comm_info(const RaynContext* ctx, int32_t* rank, int32_t* world); /* world 0 = no communicator */
/* the shard of `rank`: ascending tile indices with (tile_x + tile_y) % world == rank.  Returns the count (or the
 * needed capacity if cap is too small / out is NULL); < 0 on bad arguments.  Pure host arithmetic.                */
int32_t rayn_b200_shard_tiles(int32_t width, int32_t height, int32_t tile_w, int32_t tile_h, int32_t rank,
                              int32_t world, int32_t* out, int32_t cap);
/* render_frame for a context that holds a communicator: renders this rank's shard (frame->tile_list / tile_offset /
 * tile_stride are ignored), then all-gathers, so EVERY rank ends with the complete film in `out`, bit-identical to
 * the 1-GPU film.  Pack, ncclAllGather and unpack are enqueued on the render stream: no host synchronisation
 * between render and gather.  DEVICE planes must be non-NULL for all four channels.                               */
int32_t rayn_b200_render_frame_sharded(RaynContext* ctx, const RaynFrameDesc* frame, const RaynFilmPlanes* out);
/* the gather alone, for planes already rendered with the rank's shard (device pointers, asynchronous on the context's
 * stream; rayn_b200_sync waits).                                                                                  */
int32_t rayn_b200_film_gather(RaynContext* ctx, int32_t width, int32_t height, int32_t tile_w, int32_t tile_h,
                              const RaynFilmPlanes* planes_dev);
int32_t rayn_b200_sync(RaynContext* ctx);
/* one process driving n GPUs (contexts from comm_init_all, same scene uploaded to each): renders all shards
 * concurrently, gathers, and returns the film of ctxs[0] in `out` (HOST planes).  frame inputs must be HOST pointers. */
int32_t rayn_b200_render_frame_multi(RaynContext* const* ctxs, int32_t n, const RaynFrameDesc* frame,
                                     const RaynFilmPlanes* out);

/* ---- explicit slab helpers (device pointers): what the gather is made of; kept for hosts that bring their own
 * transport.  pack: copies the listed tiles out of full-size planes into a dense slab
 *       [n_tiles][10][tile_w*tile_h] (channel order: color rgb, alpha, bg rgb, normal xyz)
 * unpack: scatters one rank's slab back into full-size planes.                           */
int64_t rayn_b200_film_slab_floats(int32_t tile_w, int32_t tile_h, int32_t n_tiles);
/* tile_list: HOST pointer to n_tiles tile indices (the shard whose slab this is) */
int32_t rayn_b200_film_pack_tiles(RaynContext* ctx, int32_t width, int32_t height, int32_t tile_w,
                                  int32_t tile_h, const int32_t* tile_list, int32_t n_tiles,
                                  const RaynFilmPlanes* planes_dev, float* slab_dev);
int32_t rayn_b200_film_unpack_tiles(RaynContext* ctx, int32_t width, int32_t height, int32_t tile_w,
                                    int32_t tile_h, const int32_t* tile_list, int32_t n_tiles,
                                    const float* slab_dev, const RaynFilmPlanes* planes_dev);

/* ---- film post-process: the per-pixel arithmetic of Film::save_to (src/film.rs:205-377) -----
 * (SURVEY §8f rank 3: the step AFTER the path; PNG encoding itself stays host I/O.)
 * Writes the pixel buffer the reference hands to the `image` crate: rows top to bottom
 * (y flipped, film.rs:236), 8 bits per sample, `(v*255).min(255).max(0) as u8`.             */
typedef enum RaynPostMode {
  RAYN_POST_COLOR_PLUS_BACKGROUND = 0, /* RGB8  (col+bg).saturated().gamma_corrected(2.2)  film.rs:253-274 */
  RAYN_POST_COLOR_ALPHA = 1,           /* RGBA8 col.saturated().gamma_corrected(2.2), a    film.rs:230-252 */
  RAYN_POST_COLOR_ONLY = 2,            /* RGB8  col.gamma_corrected(2.2)  (no saturate)    film.rs:275-293 */
  RAYN_POST_BACKGROUND = 3,            /* RGB8  bg.saturated().gamma_corrected(2.2)        film.rs:300-325 */
  RAYN_POST_WORLD_NORMAL = 4,          /* RGB8  n*0.5 + 0.5                                film.rs:326-350 */
  RAYN_POST_ALPHA = 5                  /* L8    a                                          film.rs:351-372 */
} RaynPostMode;
/* planes->space says where the float planes live; out_space where `out` lives (RaynMemSpace).
 * out holds width*height*{3,4,3,3,3,1} bytes.                                                */
int32_t rayn_b200_film_postprocess(RaynContext* ctx, int32_t mode, int32_t width, int32_t height,
                                   const RaynFilmPlanes* planes, uint8_t* out, int32_t out_space);

/* ---- host-side input builders (pure CPU; stand in for crates the Rust host owns) ----
 * quasi-rd R_d tables (sampler.rs:18-37), rand SmallRng scramble (film.rs:460-461),
 * FilterImportanceSampler::new(BlackmanHarris) (filter.rs:13-49,196-218).               */
int32_t rayn_b200_host_rd_tables(int32_t spp, int32_t sets_1d, int32_t sets_2d, uint64_t offset,
                                 float* out_1d, float* out_2d);
int32_t rayn_b200_host_scramble(int32_t width, int32_t height, float* out);
int32_t rayn_b200_host_fis_blackman_harris(float radius, float* out512);
/* the same tables / scramble plane generated directly in device memory (DEVICE pointers; bit-identical
 * to the host builders) - saves uploading W*H floats of scramble per frame (133 MB at 8K)           */
int32_t rayn_b200_device_frame_inputs(RaynContext* ctx, int32_t width, int32_t height, int32_t spp, int32_t sets_1d,
                                      int32_t sets_2d, uint64_t offset, float* out_1d_dev, float* out_2d_dev,
                                      float* scramble_dev);
/* tile count per film.rs:399-404 (including its partial-tile quirk) */
int32_t rayn_b200_host_tile_grid(int32_t width, int32_t height, int32_t tile_w, int32_t tile_h,
                                 int32_t* n_tiles_x, int32_t* n_tiles_y);

/* ---- kernel-level known-answer entry points (device execution, host pointers) -------
 * Used by tests to compare single stages against the oracle lane by lane.              */
/* op: 0 exp, 1 ln, 2 pow(a,b), 3 sin, 4 cos, 5 tan, 6 atan2(a,b), 7 powi5               */
int32_t rayn_b200_kat_detmath(RaynContext* ctx, int32_t op, int64_t n, const float* a,
                              const float* b, float* out);
/* SDF::dist (sdf.rs:125-141) */
int32_t rayn_b200_kat_sdf_dist(RaynContext* ctx, const RaynHitable* sdf, int64_t n,
                               const float* points3, float* out);
/* the same through the packed two-point estimator the march kernels run (rt_sdf2.cuh); variant < 0 = the one the
 * scheduler would pick for this hitable, else force 0 generic Mandelbox / 1 12-iteration fast / 2 n-iteration fast / 3 Mandelbulb /
 * 4, 5 = 1, 2 with the three-operation sphere-fold division (RAYN_ERR_INVALID_ARG unless its exhaustive check passes here) */
int32_t rayn_b200_kat_sdf_dist2(RaynContext* ctx, const RaynHitable* sdf, int32_t variant, int64_t n,
                                const float* points3, float* out);
/* Newton division of the Mandelbox sphere fold vs IEEE division: number of x among the n consecutive floats starting
 * at bit pattern first_bits for which num / x differs (must be 0 wherever the fast variants are selected)           */
int32_t rayn_b200_kat_fastdiv(RaynContext* ctx, float num, uint32_t first_bits, int64_t n, int64_t* out_mismatches);
/* TracedSDF::hit (sdf.rs:59-83).  thr(t) = thr_scale * t, or thr_scale if thr_const != 0 */
int32_t rayn_b200_kat_sdf_hit(RaynContext* ctx, const RaynHitable* sdf,
                              const RaynRenderConsts* consts, int64_t n, const float* origins3,
                              const float* dirs3, const float* t_max, float thr_scale,
                              int32_t thr_const, float* out_t);
/* HitableStore::test_occluded over the uploaded scene (hitable.rs:164-168) */
int32_t rayn_b200_kat_occluded(RaynContext* ctx, int64_t n, const float* start3,
                               const float* end3, float* out);
/* HitableStore::add_hits closest-hit fold over the uploaded scene (hitable.rs:170-198):
 * out_t[i], out_obj[i] (-1 = nothing hit).  depth selects the threshold closure
 * (film.rs:540-551).                                                                     */
int32_t rayn_b200_kat_closest_hit(RaynContext* ctx, int32_t depth, int64_t n,
                                  const float* origins3, const float* dirs3, float* out_t,
                                  int32_t* out_obj);

/* SphereLight::sample (light.rs:38-72) and ::sample_volume_scattering (:75-102) per lane */
int32_t rayn_b200_kat_light_sample(RaynContext* ctx, const RaynLight* light, int64_t n, const float* s0,
                                   const float* s1, const float* points3, float* out_point3, float* out_pdf);
int32_t rayn_b200_kat_light_sample_volume(RaynContext* ctx, const RaynLight* light, int64_t n,
                                          const float* sample, const float* origins3, const float* dirs3,
                                          const float* t_max, float* out_t, float* out_pdf);
/* BSDF::scatter + BSDF::f (material.rs): normals3/wo3 unit vectors, s1d[n], u4[4n] ->
 * out_wi3, out_f3 (scatter event f), out_pdf, out_feval3 = bsdf.f(wo, wi, n) as integrator.rs:230 calls it */
int32_t rayn_b200_kat_bsdf(RaynContext* ctx, const RaynMaterial* mat, int64_t n, const float* normals3,
                           const float* wo3, const float* s1d, const float* u4, float* out_wi3,
                           float* out_f3, float* out_pdf, float* out_feval3);

/* Which march-kernel specialisation upload_scene selected for hitable `hitable_index` of the current scene: -1 analytic sphere,
 * 0 generic Mandelbox, 1 / 2 packed Mandelbox (12 / n iterations), 3 Mandelbulb, 4 / 5 = 1 / 2 with the three-operation
 * sphere-fold division, which upload_scene selects only after dividing by EVERY float in [min_rad_sq, fixed_rad_sq] on this
 * device and finding all quotients equal to IEEE division; -2 = bad index / no scene                                      */
int32_t rayn_b200_debug_sdf_variant(const RaynContext* ctx, int32_t hitable_index);

/* Packet-order debugging (SURVEY F6): when enabled, render_frame records for every depth
 * and tile the shading queue (path id per slot, -1 = padding) into an internal host log. */
int32_t rayn_b200_debug_enable_queue_log(RaynContext* ctx, int32_t enable);
/* returns number of int32 entries; copies up to cap entries.
 * Layout: repeated records { depth, tile_index, n_slots, slot[0..n_slots) }.             */
int64_t rayn_b200_debug_read_queue_log(RaynContext* ctx, int32_t* out, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* RAYN_B200_H */
