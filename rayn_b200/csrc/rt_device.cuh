// rt_device.cuh — per-lane device functions of the wavefront path tracer (sm_100a).
//
// One CUDA thread plays one lane of a reference f32x4 packet.  Every function cites the
// reference code whose per-lane behaviour it reproduces; SURVEY §9.1/9.2 argue why a
// per-lane early exit is equivalent to the reference's masked 4-lane loops.
//
// Arithmetic contract (see detmath.h): compiled with --fmad=false -prec-div=true
// -prec-sqrt=true -ftz=false, so the only fused operations are the explicit dm::fma calls
// standing where the reference writes `mul_add` (or where ultraviolet's dot/cross do).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rayn_b200.h"
#include "detmath.h"

#define RT_D __device__ __forceinline__

namespace rt {

struct f3 {
  float x, y, z;
};
RT_D f3 mk3(float x, float y, float z) { return {x, y, z}; }
RT_D f3 ld3(const float* p) { return {p[0], p[1], p[2]}; }
RT_D f3 operator+(f3 a, f3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
RT_D f3 operator-(f3 a, f3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
RT_D f3 operator*(f3 a, f3 b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }
RT_D f3 operator*(f3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
RT_D f3 operator/(f3 a, float s) { return {a.x / s, a.y / s, a.z / s}; }
RT_D f3 operator-(f3 a) { return {-a.x, -a.y, -a.z}; }
RT_D f3 fma3(f3 a, f3 b, f3 c) { return {dm::mul_add(a.x, b.x, c.x), dm::mul_add(a.y, b.y, c.y), dm::mul_add(a.z, b.z, c.z)}; }
RT_D f3 fma3s(f3 a, float s, f3 c) { return {dm::mul_add(a.x, s, c.x), dm::mul_add(a.y, s, c.y), dm::mul_add(a.z, s, c.z)}; }
// ultraviolet Wec3::dot / mag / normalized / cross / reflected (oracle/README.md A1-A5)
RT_D float dot(f3 a, f3 b) { return dm::mul_add(a.x, b.x, dm::mul_add(a.y, b.y, a.z * b.z)); }
RT_D float mag_sq(f3 a) { return dot(a, a); }
RT_D float mag(f3 a) { return sqrtf(dot(a, a)); }
RT_D f3 normalized(f3 a) {
  float r = 1.0f / mag(a);
  return a * r;
}
RT_D f3 cross(f3 a, f3 b) {
  return {dm::mul_add(a.y, b.z, -(a.z * b.y)), dm::mul_add(a.z, b.x, -(a.x * b.z)), dm::mul_add(a.x, b.y, -(a.y * b.x))};
}
RT_D f3 reflected(f3 v, f3 n) { return v - n * (2.0f * dot(v, n)); }
RT_D float component_max(f3 a) { return dm::max(dm::max(a.x, a.y), a.z); }
RT_D bool any_nan(f3 a) { return a.x != a.x || a.y != a.y || a.z != a.z; }

struct m3 {
  f3 c0, c1, c2;
};
RT_D f3 mul(const m3& m, f3 v) { return m.c0 * v.x + m.c1 * v.y + m.c2 * v.z; }

#define RT_PI 3.14159265358979323846f
#define RT_TWO_PI 6.28318530717958647692f
#define RT_FRAC_PI_2 1.57079632679489661923f
#define RT_FRAC_PI_4 0.78539816339744830962f
#define RT_EPSILON 1.1920929e-7f

// math.rs:49-59 OrthonormalBasis
RT_D m3 onb(f3 nor) {
  float ks = dm::signum(nor.z);
  float ka = 1.0f / (1.0f + dm::abs(nor.z));
  float kb = -ks * nor.x * nor.y * ka;
  f3 uu = {1.0f - nor.x * nor.x * ka, ks * kb, -ks * nor.x};
  f3 vv = {kb, ks - nor.y * nor.y * ka * ks, -nor.y};
  return {uu, vv, nor};
}

// math.rs:201-219 concentric_circle_map
RT_D void concentric(float u0, float u1, float* ox, float* oy) {
  float a = dm::mul_add(u0, 2.0f, -1.0f);
  float b = dm::mul_add(u1, 2.0f, -1.0f);
  if (a == 0.0f && b == 0.0f) b = 0.0001f;
  float phi1 = RT_FRAC_PI_4 * b / a;
  float phi2 = dm::mul_add(-RT_FRAC_PI_4 / b, a, RT_FRAC_PI_2);
  bool mask = (a * a) > (b * b);
  float r = mask ? a : b;
  float phi = mask ? phi1 : phi2;
  float s, c;
  dm::sincos(phi, &s, &c);
  *ox = r * c;
  *oy = r * s;
}
// math.rs:99-103
RT_D f3 cosine_weighted(float u0, float u1) {
  float x, y;
  concentric(u0, u1, &x, &y);
  float msq = dm::mul_add(x, x, y * y);
  float z = sqrtf(1.0f - dm::min(msq, 1.0f));
  return {x, y, z};
}
// math.rs:106-113
RT_D f3 cosine_power(float u0, float u1, float power) {
  float a = dm::pow(u0, 1.0f / (power + 1.0f));
  float a2 = a * a;
  float b = sqrtf(1.0f - a2);
  float s, c;
  dm::sincos(2.0f * u1, &s, &c);
  return {b * c, b * s, a};
}
// math.rs:122-124
RT_D float f_schlick(float cosv, float f0) { return f0 + (1.0f - f0) * dm::powi5(1.0f - cosv); }

// ------------------------------------------------------------------------------------------
// Scene as a kernel-parameter block (constant bank: warp-uniform operands cost no load)
// ------------------------------------------------------------------------------------------
// Scenes with at most SCENE_INLINE_MAX hitables, materials and lights ride in the parameter block itself (DevScene); larger
// ones keep the same tables in device memory (TableScene).  The kernels are templates on the scene type and read both
// through the same expressions (sc.hit[i], sc.sph[k], ...).
#define SCENE_INLINE_MAX 16
struct DevScene {
  static constexpr int kMaxHit = SCENE_INLINE_MAX;  // row stride - 1 of the per-tile bin tables (PassBufs::bin_start)
  int32_t n_hit, n_mat, n_lights;
  float one;  // 1.0f, set at upload: a multiplier the compiler cannot constant-fold (rt_sdf2.cuh::muladd2)
  RaynHitable hit[SCENE_INLINE_MAX];
  RaynMaterial mat[SCENE_INLINE_MAX];
  RaynLight light[SCENE_INLINE_MAX];
  RaynCamera cam;
  RaynVolume vol;
  RaynRenderConsts rc;
  // derived at upload (api.cu::rayn_b200_upload_scene): the analytic spheres and the SDF hitables as compact lists in
  // insertion order, so that the shading kernels neither walk all hitables testing `kind` nor index 40-byte descriptors per lane
  int32_t n_sph, n_sdf, sph_moving, pad_;
  int32_t sph_idx[SCENE_INLINE_MAX];  // hitable index of sphere k
  int32_t sdf_idx[SCENE_INLINE_MAX];  // hitable index of SDF ordinal j
  int32_t hit_ord[SCENE_INLINE_MAX];  // hitable i is the hit_ord[i]-th sphere / SDF
  float4 sph[SCENE_INLINE_MAX];       // centre.xyz, radius of sphere k (a moving sphere keeps its t = 0 centre here)
};

// One element of a read-only device table through the non-coherent path (LDG.CONSTANT), in the widest loads its size allows.
template <class T>
RT_D T ldg_elem(const T* p) {
  static_assert(sizeof(T) % 4 == 0, "table elements are made of 32-bit words");
  if constexpr (sizeof(T) % 16 == 0) {
    union { T t; float4 w[sizeof(T) / 16]; } u;
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 16); ++i) u.w[i] = __ldg(reinterpret_cast<const float4*>(p) + i);
    return u.t;
  } else if constexpr (sizeof(T) % 8 == 0) {
    union { T t; float2 w[sizeof(T) / 8]; } u;
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 8); ++i) u.w[i] = __ldg(reinterpret_cast<const float2*>(p) + i);
    return u.t;
  } else {
    union { T t; float w[sizeof(T) / 4]; } u;
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 4); ++i) u.w[i] = __ldg(reinterpret_cast<const float*>(p) + i);
    return u.t;
  }
}
template <class T>
struct LdgTable {
  const T* p;
  RT_D T operator[](int i) const { return ldg_elem(p + i); }
};
// The scene of the large-scene path: DevScene's fields, its arrays as tables in device memory that the context owns
// (written once per upload, api.cu).  Loads that differ per lane (the hit object's descriptor, its material, a light) and
// the loops every lane of a warp walks in the same order (sphere lists) both go through LDG: the uniform ones are one
// broadcast transaction per warp, served from L1 after the first warp of the SM.
struct TableScene {
  static constexpr int kMaxHit = RAYN_MAX_HITABLES;
  int32_t n_hit, n_mat, n_lights;
  float one;
  LdgTable<RaynHitable> hit;
  LdgTable<RaynMaterial> mat;
  LdgTable<RaynLight> light;
  RaynCamera cam;
  RaynVolume vol;
  RaynRenderConsts rc;
  int32_t n_sph, n_sdf, sph_moving, pad_;
  LdgTable<int32_t> sph_idx, sdf_idx, hit_ord;
  LdgTable<float4> sph;
};

// the `hit_threshold_at` closure of film.rs:540-551
struct Thr {
  float scale;
  int is_const;
  RT_D float at(float t) const { return is_const ? scale : scale * t; }
};
__host__ __device__ inline Thr make_thr(const RaynCamera& cam, int depth) {
  Thr t;
  if (depth == 0) {
    t.scale = cam.half_pixel_size;                               // camera.rs:116-118,210-212
    t.is_const = cam.kind == RAYN_CAMERA_ORTHOGRAPHIC ? 1 : 0;  // camera.rs:282-284
  } else {
    t.scale = 0.0001f * 2.0f * (float)depth;  // film.rs:549
    t.is_const = 0;
  }
  return t;
}

// ---- SDFs ----------------------------------------------------------------------------------
// A distance evaluation is kept as an explicit little state machine (start / more / step /
// finish) so that the eval-granular kernels and the iteration-granular ("flattened") march
// kernels execute literally the same arithmetic.
//   MandelBox::dist, sdf.rs:125-141 (+ BoxFold :160-162, SphereFold :181-187):
//     w = running point, c = offset (the original point), dr, it.
//   Mandelbulb (AUTHORED, no reference counterpart; SURVEY F1; definition in DESIGN.md):
//     w, c, dr, m = |w|^2, it; stops early once m > bailout^2.
struct SdfEval {
  f3 w, c;
  float dr, m;
  int it;
};
RT_D void eval_start(SdfEval& e, const RaynHitable& h, f3 p) {
  e.w = p;
  e.c = p;
  e.dr = 1.0f;
  e.it = 0;
  e.m = h.kind == RAYN_HITABLE_MANDELBULB ? dot(p, p) : 0.0f;
}
RT_D bool eval_more(const SdfEval& e, const RaynHitable& h) {
  if (h.kind == RAYN_HITABLE_MANDELBULB) return e.it < h.iterations && !(e.m > h.bulb_bailout * h.bulb_bailout);
  return e.it < h.iterations;
}
RT_D void eval_step(SdfEval& e, const RaynHitable& h) {
  if (h.kind == RAYN_HITABLE_MANDELBULB) {
    const f3 w = e.w;
    const float m = e.m;
    const float m2 = m * m, m3 = m2 * m;
    const float r = sqrtf(m);
    const float r7 = m3 * r;
    e.dr = dm::fma(8.0f * r7, e.dr, 1.0f);
    const float a = w.z * w.z, b = m;
    const float b2 = b * b, b3 = b2 * b, b4 = b2 * b2;
    // Horner forms with explicit fused multiply-adds (the definition is ours: DESIGN.md §7)
    const float P = dm::fma(dm::fma(dm::fma(dm::fma(128.0f, a, -256.0f * b), a, 160.0f * b2), a, -32.0f * b3), a, b4);
    const float A = dm::fma(dm::fma(dm::fma(128.0f, a, -192.0f * b), a, 80.0f * b2), a, -8.0f * b3);
    const float ax = w.x * w.x;
    const float q = dm::fma(w.x, w.x, w.y * w.y);
    const float q2 = q * q, q3 = q2 * q, q4 = q2 * q2;
    const float C = dm::fma(dm::fma(dm::fma(dm::fma(128.0f, ax, -256.0f * q), ax, 160.0f * q2), ax, -32.0f * q3), ax, q4);
    const float B = dm::fma(dm::fma(dm::fma(128.0f, ax, -192.0f * q), ax, 80.0f * q2), ax, -8.0f * q3);
    float k = (w.z * A) / (q3 * sqrtf(q));
    k = q > 0.0f ? k : 0.0f;
    e.w = mk3(dm::fma(k, C, e.c.x), dm::fma(k, w.x * w.y * B, e.c.y), P + e.c.z);
    e.m = dot(e.w, e.w);
  } else {
    const float l = h.box_l, nl = -h.box_l;
    f3 p = e.w;
    // clamped(neg_l, l) = max(neg_l).min(l), then mul_add(two, -p).  SSE maxps/minps return the SECOND operand when
    // unordered; with a constant, non-NaN, non-zero second operand that is exactly fmaxf/fminf for every input
    // (NaN -> the constant either way; no signed-zero tie is possible), so one FMNMX replaces compare + select.
    float cx, cy, cz;
    if (l > 0.0f) {
      cx = fminf(fmaxf(p.x, nl), l);
      cy = fminf(fmaxf(p.y, nl), l);
      cz = fminf(fmaxf(p.z, nl), l);
    } else {
      cx = dm::min(dm::max(p.x, nl), l);
      cy = dm::min(dm::max(p.y, nl), l);
      cz = dm::min(dm::max(p.z, nl), l);
    }
    p.x = dm::mul_add(cx, 2.0f, -p.x);
    p.y = dm::mul_add(cy, 2.0f, -p.y);
    p.z = dm::mul_add(cz, 2.0f, -p.z);
    const float r2 = mag_sq(p);
    const float mul = dm::max(1.0f, h.fixed_rad_sq / dm::max(h.min_rad_sq, r2));
    p = p * mul;
    e.dr = e.dr * mul;
    e.w = fma3s(p, h.scale, e.c);
    e.dr = dm::mul_add(-e.dr, h.scale, 1.0f);
  }
  ++e.it;
}
RT_D float eval_finish(const SdfEval& e, const RaynHitable& h) {
  if (h.kind == RAYN_HITABLE_MANDELBULB) {
    const float r = sqrtf(e.m);
    return 0.5f * dm::ln_fast(r) * r / e.dr;
  }
  return mag(e.w) / dm::abs(e.dr);
}
RT_D float sdf_dist(const RaynHitable& h, f3 p) {
  SdfEval e;
  eval_start(e, h, p);
  while (eval_more(e, h)) eval_step(e, h);
  return eval_finish(e, h);
}

// TracedSDF::hit per lane, sdf.rs:59-83 / SURVEY §9.1.  *evals counts dist() calls.
RT_D float sdf_hit(const RaynHitable& h, const RaynRenderConsts& rc, f3 o, f3 d, float t_max, Thr thr, int* evals) {
  float t = sdf_dist(h, o);
  *evals += 1;
  if (t != t) return t;
  const float S = rc.sdf_detail_scale;
  const float c0 = 0.00005f * S, c1 = 0.05f * S;
  for (int march = 0; march < rc.max_marches; ++march) {
    f3 p = fma3s(d, t, o);
    float dd = sdf_dist(h, p);
    *evals += 1;
    bool hit = dm::abs(dd) < dm::max(c0, c1 * thr.at(t));
    bool gt = t > t_max;
    if (hit || gt) break;
    t = t + dd;
    if (t != t) break;  // NaN can never satisfy hit/gt again: marches to exhaustion, returns NaN
  }
  return t;
}

// TracedSDF::occluded per lane, sdf.rs:25-57 / SURVEY §9.2.  1 = visible, 0 = occluded.
RT_D float sdf_occluded(const RaynHitable& h, const RaynRenderConsts& rc, f3 start, f3 end, int* evals) {
  f3 dir = end - start;
  float max_dist = mag(dir);
  dir = dir / max_dist;
  float t = sdf_dist(h, start);
  *evals += 1;
  if (t != t) return 1.0f;
  const float S = rc.sdf_detail_scale;
  const float c0 = 0.0001f * S, c1 = 0.00001f * S;
  for (int march = 0; march < rc.max_vis_marches; ++march) {
    if (t > max_dist) return 1.0f;
    f3 p = fma3s(dir, t, start);
    float dd = sdf_dist(h, p);
    *evals += 1;
    if (dm::abs(dd) < dm::max(c0, c1 * t)) return 0.0f;
    t = t + dd;
    if (t != t) return 1.0f;
  }
  return 1.0f;
}

// ---- Sphere, sphere.rs ------------------------------------------------------------------------
// WSequenced<Wec3>::sample_at for the sphere centre.  A non-zero velocity stands for the closure
// `|t| center + velocity * t`, which the reference evaluates at LANE 0's time of the 4-lane packet
// (animation.rs:62-67): `time0` is that time.  Zero velocity = constant (animation.rs:52).
RT_D f3 seq3(const float* base, const float* vel, float time0) {
  f3 c = ld3(base);
  const f3 v = ld3(vel);
  if (v.x != 0.0f || v.y != 0.0f || v.z != 0.0f) c = c + v * time0;
  return c;
}
RT_D f3 sphere_center(const RaynHitable& h, float time0) { return seq3(h.center, h.center_velocity, time0); }
RT_D bool sphere_moves(const RaynHitable& h) {
  return h.kind == RAYN_HITABLE_SPHERE && (h.center_velocity[0] != 0.0f || h.center_velocity[1] != 0.0f || h.center_velocity[2] != 0.0f);
}
// Sphere::occluded, sphere.rs:24-46, with the segment's direction and length (lines :25-27: `dir = end - start; dist = dir.mag();
// dir /= dist`) computed ONCE by the caller: they are the same expressions for every hitable of a segment (TracedSDF::occluded
// starts with the same three lines, sdf.rs:26-28), so hoisting them changes no bit.
RT_D float sphere_occluded_seg(const RaynHitable& h, f3 start, f3 dir, float dist, float time0) {
  f3 oc = start - sphere_center(h, time0);
  float b = dot(oc, dir);
  float c = mag_sq(oc) - h.radius * h.radius;
  float descrim = b * b - c;
  bool desc_pos = descrim > 0.0f;
  float desc_sqrt = sqrtf(descrim);
  float t1 = -b - desc_sqrt;
  float t2 = -b + desc_sqrt;
  float mn = dm::min(t1, t2);
  bool valid = (mn > 0.001f) && (t1 <= dist) && desc_pos;
  return valid ? 0.0f : 1.0f;
}
// The same for a STATIC sphere given as (centre, radius).  sqrt is skipped when the discriminant is not positive (or NaN):
// `valid` is false then whatever the root would have been, so the result is the same 1.0.
RT_D float sphere_occluded_seg_static(const float4 cr, f3 start, f3 dir, float dist) {
  const f3 oc = start - mk3(cr.x, cr.y, cr.z);
  const float b = dot(oc, dir);
  const float c = mag_sq(oc) - cr.w * cr.w;
  const float descrim = b * b - c;
  if (!(descrim > 0.0f)) return 1.0f;
  const float desc_sqrt = sqrtf(descrim);
  const float t1 = -b - desc_sqrt;
  const float t2 = -b + desc_sqrt;
  const float mn = dm::min(t1, t2);
  const bool valid = (mn > 0.001f) && (t1 <= dist);
  return valid ? 0.0f : 1.0f;
}
RT_D float sphere_occluded(const RaynHitable& h, f3 start, f3 end, float time0) {  // :24-46
  f3 dir = end - start;
  float dist = mag(dir);
  dir = dir / dist;
  f3 oc = start - sphere_center(h, time0);
  float b = dot(oc, dir);
  float c = mag_sq(oc) - h.radius * h.radius;
  float descrim = b * b - c;
  bool desc_pos = descrim > 0.0f;
  float desc_sqrt = sqrtf(descrim);
  float t1 = -b - desc_sqrt;
  float t2 = -b + desc_sqrt;
  float mn = dm::min(t1, t2);
  bool valid = (mn > 0.001f) && (t1 <= dist) && desc_pos;
  return valid ? 0.0f : 1.0f;
}
RT_D float sphere_hit(const RaynHitable& h, f3 ro, f3 rd, float t_max, float time0) {  // :48-72
  f3 oc = ro - sphere_center(h, time0);
  float b = dot(oc, rd);
  float c = mag_sq(oc) - h.radius * h.radius;
  float descrim = b * b - c;
  bool desc_pos = descrim > 0.0f;
  float desc_sqrt = sqrtf(descrim);
  float t1 = -b - desc_sqrt;
  bool t1_valid = (t1 > 0.0001f) && (t1 <= t_max) && desc_pos;
  float t2 = -b + desc_sqrt;
  bool t2_valid = (t2 > 0.0001f) && (t2 <= t_max) && desc_pos;
  bool take_t1 = (t1 < t2) && t1_valid;
  float t = take_t1 ? t1 : t2;
  return (t1_valid || t2_valid) ? t : 3.40282347e+38f;
}

// Sphere::hit for a STATIC sphere given as (centre, radius): no root is taken when the discriminant is not positive (or NaN),
// both candidates are invalid then and the result is the same f32::MAX.
RT_D float sphere_hit_static(const float4 cr, f3 ro, f3 rd, float t_max) {
  const f3 oc = ro - mk3(cr.x, cr.y, cr.z);
  const float b = dot(oc, rd);
  const float c = mag_sq(oc) - cr.w * cr.w;
  const float descrim = b * b - c;
  if (!(descrim > 0.0f)) return 3.40282347e+38f;
  const float desc_sqrt = sqrtf(descrim);
  const float t1 = -b - desc_sqrt;
  const bool t1_valid = (t1 > 0.0001f) && (t1 <= t_max);
  const float t2 = -b + desc_sqrt;
  const bool t2_valid = (t2 > 0.0001f) && (t2 <= t_max);
  const bool take_t1 = (t1 < t2) && t1_valid;
  const float t = take_t1 ? t1 : t2;
  return (t1_valid || t2_valid) ? t : 3.40282347e+38f;
}

// HitableStore::add_hits fold, hitable.rs:177-198
template <class Scn>
RT_D void closest_hit(const Scn& sc, f3 o, f3 d, Thr thr, float* out_t, int* out_obj, int* evals, float time0 = 0.0f) {
  float closest = sc.rc.world_radius * 2.0f;  // film.rs:556
  int id = -1;
  for (int i = 0; i < sc.n_hit; ++i) {
    const RaynHitable& h = sc.hit[i];
    float t = h.kind == RAYN_HITABLE_SPHERE ? sphere_hit(h, o, d, closest, time0) : sdf_hit(h, sc.rc, o, d, closest, thr, evals);
    if (t < closest) {
      closest = t;
      id = i;
    }
  }
  *out_t = closest;
  *out_obj = id;
}

// HitableStore::test_occluded, hitable.rs:164-168.  The reference multiplies occluded() in
// {0,1} over ALL hitables; a product of exact 0/1 floats is 0 iff any factor is 0, so the
// cheap analytic spheres are tested first and the march is skipped once occlusion is known.
template <class Scn>
RT_D float test_occluded(const Scn& sc, f3 start, f3 end, int* evals, float time0 = 0.0f) {
  for (int i = 0; i < sc.n_hit; ++i)
    if (sc.hit[i].kind == RAYN_HITABLE_SPHERE && sphere_occluded(sc.hit[i], start, end, time0) == 0.0f) return 0.0f;
  for (int i = 0; i < sc.n_hit; ++i)
    if (sc.hit[i].kind != RAYN_HITABLE_SPHERE && sdf_occluded(sc.hit[i], sc.rc, start, end, evals) == 0.0f) return 0.0f;
  return 1.0f;
}

// ---- shading info --------------------------------------------------------------------------------
struct ShadingPoint {  // hitable.rs:21-28 (per lane)
  f3 o, d;             // the incoming ray
  float time, t;
  f3 point;
  float offset_by;
  f3 normal;
  m3 basis;
};
// sdf.rs:85-101 with sdfu's tetrahedral normals_fast (oracle/README.md A8); sphere.rs:74-86
RT_D void shading_info(const DevScene& sc, const RaynHitable& h, Thr thr, ShadingPoint& sp, int* evals, bool want_basis = true,
                       float time0 = 0.0f) {
  sp.point = fma3s(sp.d, sp.t, sp.o);  // WHit::point -> ray.point_at, ray.rs:22-24
  if (h.kind == RAYN_HITABLE_SPHERE) {
    sp.normal = normalized(sp.point - sphere_center(h, time0));
    sp.offset_by = 0.0f;
  } else {
    float eps = dm::max(0.0001f, sc.rc.sdf_detail_scale * thr.at(sp.t));
    // tetrahedron offsets xyy, yyx, yxy, xxx in that order; rolled loop (one inlined copy of the distance
    // estimator instead of four: the kernel was stalling on instruction fetch), same left-to-right sum
    f3 n = {0.0f, 0.0f, 0.0f};
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
      const f3 k = {(i == 0 || i == 3) ? 1.0f : -1.0f, (i == 2 || i == 3) ? 1.0f : -1.0f, (i == 1 || i == 3) ? 1.0f : -1.0f};
      const float d = sdf_dist(h, sp.point + k * eps);
      n = i == 0 ? k * d : n + k * d;
    }
    *evals += 4;
    sp.normal = normalized(n);
    sp.offset_by = eps;
  }
  if (want_basis) sp.basis = onb(sp.normal);
}

// ---- lights, light.rs ---------------------------------------------------------------------------
RT_D void light_sample(const RaynLight& L, float s0, float s1, f3 p, f3* out_point, f3* out_li, float* out_pdf) {  // :38-72
  f3 pos = ld3(L.pos);
  float rad = L.rad;
  f3 dir_to_light = pos - p;
  float dist_sq = mag_sq(dir_to_light);
  float dist = sqrtf(dist_sq);
  dir_to_light = dir_to_light / dist;
  m3 basis = onb(-dir_to_light);
  float r2 = rad * rad;
  float sin_theta_max_2 = r2 / dist_sq;
  float cos_theta_max = sqrtf(dm::max(0.0f, 1.0f - sin_theta_max_2));
  float cos_theta = (1.0f - s0) + s0 * cos_theta_max;
  float sin_theta = sqrtf(dm::max(0.0f, 1.0f - cos_theta * cos_theta));
  float phi = s1 * RT_TWO_PI;
  float ds = dist * cos_theta - sqrtf(dm::max(0.0f, r2 - dist_sq * sin_theta * sin_theta));
  float cos_alpha = (dist_sq + r2 - ds * ds) / (2.0f * dist * rad);
  float sin_alpha = sqrtf(dm::max(0.0f, 1.0f - cos_alpha * cos_alpha));
  float sin_phi, cos_phi;
  dm::sincos(phi, &sin_phi, &cos_phi);
  f3 offset = basis.c0 * sin_alpha * cos_phi + basis.c1 * sin_alpha * sin_phi + basis.c2 * cos_alpha;
  *out_point = pos + offset * rad;
  *out_li = ld3(L.emission);
  *out_pdf = 1.0f / (RT_TWO_PI * (1.0f - cos_theta_max));  // uniform_cone_pdf :105-107
}
RT_D void light_sample_volume(const RaynLight& L, float sample, f3 ray_o, f3 ray_d, float max_distance, float* out_dist,
                              float* out_pdf) {  // :75-102
  f3 pos = ld3(L.pos);
  float delta = dot(pos - ray_o, ray_d);
  f3 closest_point = ray_o + ray_d * delta;
  float d = mag(closest_point - pos);
  float theta_a = dm::atan2(-delta, d);
  float theta_b = dm::atan2(max_distance - delta, d);
  float th = theta_a * (1.0f - sample) + theta_b * sample;  // Lerp (A7)
  float t = d * dm::tan(th);
  *out_dist = delta + t;
  *out_pdf = d / ((theta_b - theta_a) * dm::mul_add(d, d, t * t));
}

// ---- BSDFs, material.rs ---------------------------------------------------------------------------
RT_D bool receives_light(const RaynMaterial& m) {
  return m.kind == RAYN_MATERIAL_LAMBERTIAN || m.kind == RAYN_MATERIAL_DIELECTRIC;
}
RT_D f3 bsdf_le(const RaynMaterial& m, f3 wo) {
  if (m.kind == RAYN_MATERIAL_SKY) {  // :444-448
    float t = 0.5f * (wo.y + 1.0f);
    return ld3(m.sky_top) * (1.0f - t) + ld3(m.sky_bottom) * t;
  }
  if (m.kind == RAYN_MATERIAL_EMISSIVE) return ld3(m.emission);  // :517-519
  return {0.0f, 0.0f, 0.0f};
}
// called as bsdf.f(wo, wi, n) (integrator.rs:230); see oracle note on argument naming.
RT_D f3 bsdf_f(const RaynMaterial& m, f3 first, f3 second, f3 n) {
  f3 albedo = ld3(m.albedo);
  if (m.kind == RAYN_MATERIAL_LAMBERTIAN) return albedo / RT_PI;  // :139-141
  float rough = m.roughness;                                      // Dielectric :195-205
  float dotv = dm::max(0.0f, dot(first, n));
  float fresnel = f_schlick(dotv, 0.04f);
  f3 half = normalized(second + first);
  float cos_alpha = dm::pow(dm::max(0.0f, dot(half, n)), rough);
  float spec_factor = cos_alpha * (rough + 2.0f) / (2.0f * RT_PI);
  f3 spec_f = mk3(1.0f, 1.0f, 1.0f) * spec_factor * fresnel;
  f3 diffuse_f = albedo / RT_PI * (1.0f - fresnel);
  return spec_f + diffuse_f;
}
struct Scatter {
  f3 wi, f;
  float pdf;
};
RT_D Scatter bsdf_scatter(const RaynMaterial& m, f3 wo, const ShadingPoint& sp, float s1d, float u0, float u1, float u2,
                          float u3) {
  Scatter se;
  if (m.kind != RAYN_MATERIAL_DIELECTRIC) {  // Lambertian :118-137 (Emissive/Sky never scatter on the path)
    f3 ds = cosine_weighted(u0, u1);
    se.wi = normalized(mul(sp.basis, ds));
    se.f = ld3(m.albedo) / RT_PI;
    se.pdf = ds.z / RT_PI;
    return se;
  }
  // Dielectric :207-256
  f3 albedo = ld3(m.albedo);
  float rough = m.roughness;
  f3 norm = sp.normal;
  float cosv = dm::abs(dot(norm, wo));
  f3 diffuse_sample = cosine_weighted(u0, u1);
  f3 diffuse_bounce = normalized(mul(sp.basis, diffuse_sample));
  float diffuse_pdf = dm::max(0.00001f, diffuse_sample.z / RT_PI);
  f3 diffuse_f = albedo / RT_PI;
  f3 spec_sample = cosine_power(u2, u3, rough);
  f3 reflection = reflected(wo, norm);
  m3 basis = onb(reflection);
  f3 spec_bounce = normalized(mul(basis, spec_sample));
  float cos_alpha_pow = dm::max(dm::pow(spec_sample.z, rough), RT_EPSILON);
  float spec_pdf = (rough + 1.0f) / RT_TWO_PI * cos_alpha_pow;
  float spec_coeff = (rough + 2.0f) / RT_TWO_PI * cos_alpha_pow;
  bool below_horizon = dot(norm, spec_bounce) < 0.0f;
  spec_coeff = below_horizon ? 0.0f : spec_coeff;
  f3 spec_f = mk3(1.0f, 1.0f, 1.0f) * spec_coeff;
  float fresnel = f_schlick(cosv, 0.04f);
  bool fresnel_mask = s1d < fresnel;
  se.wi = fresnel_mask ? spec_bounce : diffuse_bounce;
  se.f = fresnel_mask ? spec_f : diffuse_f;
  se.pdf = fresnel * spec_pdf + (1.0f - fresnel) * diffuse_pdf;
  return se;
}

RT_D int light_index(float s, int n_lights) {  // integrator.rs:76-77 (+ clamp, A10)
  int i = (int)floorf(s * (float)n_lights);
  if (i < 0) i = 0;
  if (i > n_lights - 1) i = n_lights - 1;
  return i;
}

// ---- camera.rs ---------------------------------------------------------------------------------------
// time0 = the time of lane 0 of the camera packet (the 4 samples 4k..4k+3 of one pixel), see seq3()
RT_D void camera_ray(const RaynCamera& c, float u, float v, float ls0, float ls1, float time0, f3* ro, f3* rd) {
  f3 origin = seq3(c.origin, c.origin_velocity, time0), at = seq3(c.at, c.at_velocity, time0), up = seq3(c.up, c.up_velocity, time0);
  float hx = c.half_size[0], hy = c.half_size[1];
  if (c.kind == RAYN_CAMERA_PINHOLE) {  // :81-114
    f3 bw = normalized(origin - at);
    f3 bu = normalized(cross(up, bw));
    f3 bv = cross(bw, bu);
    f3 lower_left = origin - bu * hx - bv * hy - bw;
    f3 horiz = bu * hx * 2.0f * u;
    f3 verti = bv * hy * 2.0f * v;
    *ro = origin;
    *rd = normalized(lower_left + horiz + verti - origin);
  } else if (c.kind == RAYN_CAMERA_THINLENS) {  // :168-208
    float focus_dist = mag(seq3(c.focus, c.focus_velocity, time0) - origin);
    const float aperture = c.aperture_rate == 0.0f ? c.aperture : c.aperture + c.aperture_rate * time0;
    f3 bw = normalized(origin - at);
    f3 bu = normalized(cross(up, bw));
    f3 bv = cross(bw, bu);
    f3 lower_left = origin - bu * hx * focus_dist - bv * hy * focus_dist - bw * focus_dist;
    f3 horiz = bu * hx * focus_dist * 2.0f * u;
    f3 verti = bv * hy * focus_dist * 2.0f * v;
    float dx, dy;
    concentric(ls0, ls1, &dx, &dy);
    dx = dx * aperture;
    dy = dy * aperture;
    f3 offset = bu * dx + bv * dy;
    f3 o2 = origin + offset;
    *ro = o2;
    *rd = normalized(lower_left + horiz + verti - o2);
  } else {  // orthographic :249-280
    f3 bw = normalized(at - origin);
    f3 bu = normalized(cross(bw, up));
    f3 bv = cross(bu, bw);
    f3 lower_left = origin - bu * hx - bv * hy;
    f3 offset = bu * u * c.full_size[0] + bv * v * c.full_size[1];
    *ro = lower_left + offset;
    *rd = bw;
  }
}

// filter.rs:222-235
RT_D float fis_sample(const float* __restrict__ inv, float u) {
  u = 2.0f * (u - 0.5f);
  float mult = u < 0.0f ? -1.0f : 1.0f;
  u = fminf(fmaxf(fabsf(u), 0.0f), 0.99999f);
  float idx_full = u * (float)(RAYN_FIS_TABLE_SIZE - 1);
  int idx = (int)floorf(idx_full);
  float t = dm::fract(idx_full);
  return mult * (inv[idx] * (1.0f - t) + inv[idx + 1] * t);
}

}  // namespace rt
