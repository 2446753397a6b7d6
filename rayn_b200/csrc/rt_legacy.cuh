// rt_legacy.cuh — round-1 "v0" kernels: one thread per ray (k_extend) and one thread per shading slot with the
// shadow marches fused in (k_shade).  TEST-ONLY: compiled only with -DRAYN_LEGACY_KERNELS into
// librayn_b200_legacy.so, where RAYN_FLAG_SIMPLE_MARCH selects them.  They are a structurally independent
// second implementation of the same per-lane functions (no queues of shadow segments, no lane refill, no packed
// arithmetic), which is what makes them a useful cross-check of the product kernels in tests/.
#pragma once
#include "rt_kernels.cuh"

namespace rt {

// ------------------------------------------------------------------------------------------
// K2 extend: HitableStore::add_hits (hitable.rs:170-210) incl. the sphere-march
// (sdf.rs:59-83).  One thread per live ray: reads float4 o_time + float4 d, writes t + key.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_extend(const __grid_constant__ DevScene sc, const PassBufs pb, const Thr thr) {
  const int ts = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = pb.n_live[ts];
  if ((i & ~31) >= n) return;
  int evals = 0;
  const bool act = i < n;
  if (act) {
    const size_t q = (size_t)ts * pb.R + i;
    const int id = pb.q_live[q];
    const size_t g = (size_t)ts * pb.R + id;
    const float4 o4 = pb.o_time[g];
    const float4 d4 = pb.d_t[g];
    float t;
    int obj;
    closest_hit(sc, mk3(o4.x, o4.y, o4.z), mk3(d4.x, d4.y, d4.z), thr, &t, &obj, &evals);
    pb.d_t[g].w = t;
    pb.q_key[g] = obj;
  }
  warp_add(pb.counters + CNT_EVALS_EXTEND, evals);
}

// ------------------------------------------------------------------------------------------
// K4 shade (+K5 shadow fused): get_shading_info (sdf.rs:85-101 / sphere.rs:74-86), sample
// draw (film.rs:564-589), PathTracingIntegrator::integrate (integrator.rs:47-205).
// One thread per shading slot; lanes 4k..4k+3 of a warp are exactly one reference packet and
// exchange their light choices with __shfl_sync (SURVEY §9.3).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_shade(const __grid_constant__ DevScene sc, const DevFrame fr, const PassBufs pb,
                                               const int depth, const Thr thr) {
  const int ts = blockIdx.y;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const int nslots = pb.n_slots[ts];
  if ((s & ~31) >= nslots) return;  // warp-uniform
  const int lane = threadIdx.x & 31;
  int* __restrict__ qs = pb.q_shade + (size_t)ts * pb.QS;
  const int id = s < nslots ? qs[s] : -1;
  const bool valid = id >= 0;
  const TileGeom tg = tile_geom(fr, pb.tile_ids[ts]);
  // sample index / scramble: padded lanes are Ray::new_invalid -> sample 0, scramble 0 (ray.rs:54-66)
  int sample = 0;
  float scramble = 0.0f;
  int pl = 0;
  if (valid) {
    pl = id / fr.spp;
    sample = id - pl * fr.spp;
    const int xl = pl / tg.th, yl = pl - xl * tg.th;
    scramble = __ldg(fr.scramble + (tg.x0 + xl) + (size_t)(tg.y0 + yl) * fr.W);
  }
  const int n1 = 3 + fr.vm, n2h = (12 + 8 * fr.vm) / 2;  // 1-D sets / 2-D sets per depth
  const int set1 = 1 + depth * n1, set2 = 2 + depth * n2h;
  const int nl = sc.n_lights;
  // light choices: one index per lane per light-selection sample (integrator.rs:76-77,100-102)
  unsigned pack = 0;
  if (nl > 0) {
    pack = (unsigned)light_index(samp1(fr, sample, scramble, set1 + 0), nl) |
           ((unsigned)light_index(samp1(fr, sample, scramble, set1 + 1), nl) << 8) |
           ((unsigned)light_index(samp1(fr, sample, scramble, set1 + 2), nl) << 16);
  }
  unsigned packs[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) packs[k] = __shfl_sync(0xffffffffu, pack, (lane & ~3) + k);
  warp_add(pb.counters + CNT_SHADE_LANES, valid ? 1 : 0);
  int evals = 0, shadows = 0;
  if (valid) {
    // object of this slot from the tile's bin table
    const int* __restrict__ bs = pb.bin_start + ts * (SCENE_INLINE_MAX + 1);
    int obj = 0;
    while (obj + 1 < sc.n_hit && s >= bs[obj + 1]) ++obj;
    const RaynHitable& h = sc.hit[obj];
    const RaynMaterial& mat = sc.mat[h.material];
    const size_t g = (size_t)ts * pb.R + id;
    const float4 o4 = pb.o_time[g], d4 = pb.d_t[g], r4 = pb.rad[g], t4 = pb.thr[g];
    ShadingPoint sp;
    sp.o = mk3(o4.x, o4.y, o4.z);
    sp.d = mk3(d4.x, d4.y, d4.z);
    sp.time = o4.w;
    sp.t = d4.w;
    shading_info(sc, h, thr, sp, &evals);
    f3 radiance = mk3(r4.x, r4.y, r4.z), throughput = mk3(t4.x, t4.y, t4.z);
    const f3 wo = -sp.d;
    const bool has_ext = sc.vol.has_extinction != 0;
    const float neg_rho_t = -sc.vol.coeff_extinction;
    const float vt = has_ext ? dm::exp(neg_rho_t * sp.t) : 1.0f;  // integrator.rs:64-68
    radiance = radiance + bsdf_le(mat, wo) * throughput * vt;        // :70-71
    const bool recv = receives_light(mat);

    if (recv && nl > 0) {  // :73-94
      const float correction = (float)nl / 4.0f;
#pragma unroll 1
      for (int i = 0; i < 4; ++i) {
        const int li_idx = (int)(packs[i] & 0xffu);
        const float u0 = samp2(fr, 0, sample, scramble, set2 + i), u1 = samp2(fr, 1, sample, scramble, set2 + i);
        // surface_sample_one_light :207-240
        f3 end_point, li;
        float pdf;
        light_sample(sc.light[li_idx], u0, u1, sp.point, &end_point, &li, &pdf);
        f3 wi = end_point - sp.point;
        const float dist = mag(wi);
        wi = wi / dist;
        const f3 occlude_point = sp.point + sp.normal * dm::signum(dot(sp.normal, wi)) * sp.offset_by;
        const float occluded = test_occluded(sc, occlude_point, end_point, &evals);
        ++shadows;
        const f3 f = bsdf_f(mat, wo, wi, sp.normal) * dm::max(dot(sp.normal, wi), 0.0f);
        const float transmission = has_ext ? dm::exp(neg_rho_t * dist) : 1.0f;
        const f3 contrib = li * f * transmission * occluded / pdf;
        radiance = radiance + contrib * throughput * correction * vt;
      }
    }
    if (sc.vol.has_scattering && nl > 0) {  // :96-132
      const float rho_s = sc.vol.coeff_scattering;
      const float correction = (float)nl / 4.0f / (float)fr.vm;
      const float vol_sample = samp1(fr, sample, scramble, set1 + 1);  // samples_1d[1], :115
#pragma unroll 1
      for (int march = 0; march < fr.vm; ++march) {
#pragma unroll 1
        for (int i = 0; i < 4; ++i) {
          const int li_idx = (int)((packs[i] >> (8 * (march + 1))) & 0xffu);
          const int set = set2 + 4 + 4 * march + i;  // samples_2d[8 + 8*march + 2i]
          const float u0 = samp2(fr, 0, sample, scramble, set), u1 = samp2(fr, 1, sample, scramble, set);
          // volume_sample_one_light :242-281
          const RaynLight& L = sc.light[li_idx];
          float vol_dist, vol_pdf;
          light_sample_volume(L, vol_sample, sp.o, sp.d, sp.t, &vol_dist, &vol_pdf);
          const f3 sampled_point = sp.o + sp.d * vol_dist;
          f3 end_point, li;
          float light_pdf;
          light_sample(L, u0, u1, sampled_point, &end_point, &li, &light_pdf);
          const f3 wi = end_point - sampled_point;
          const float dist_point_to_light = mag(wi);
          const float occluded = test_occluded(sc, sampled_point, end_point, &evals);
          ++shadows;
          const float f = 1.0f / (4.0f * RT_PI);
          const float tr_light = has_ext ? dm::exp(neg_rho_t * dist_point_to_light) : 1.0f;
          const f3 contrib = li * f * tr_light * occluded / (vol_pdf * light_pdf);
          const float transmission = has_ext ? dm::exp(neg_rho_t * vol_dist) : 1.0f;
          radiance = radiance + contrib * throughput * correction * rho_s * transmission;
        }
      }
    }

    if (recv) {  // :134-188
      const int setb = set2 + 4 + 4 * fr.vm;  // samples_2d[8 + 8*vm ..]
      const Scatter se = bsdf_scatter(mat, wo, sp, samp1(fr, sample, scramble, set1 + 3), samp2(fr, 0, sample, scramble, setb),
                                      samp2(fr, 1, sample, scramble, setb), samp2(fr, 0, sample, scramble, setb + 1),
                                      samp2(fr, 1, sample, scramble, setb + 1));
      const float ndl = dm::abs(dot(se.wi, sp.normal));
      f3 new_throughput = throughput * vt * se.f * ndl / se.pdf;
      float roulette_factor = 0.0f;
      if (depth > 2) {
        roulette_factor = dm::max(1.0f - component_max(throughput), 0.05f);
        new_throughput = new_throughput / (1.0f - roulette_factor);
      }
      if (depth == 0)  // Alpha(1) + WorldNormal(n), :161-169
        pb.nrm0[g] = make_float4(sp.normal.x, sp.normal.y, sp.normal.z, __uint_as_float((unsigned)s + 1u));
      const float roulette_sample = samp1(fr, sample, scramble, set1 + 4);
      if (depth >= fr.max_bounces || roulette_sample < roulette_factor) {
        pb.rad[g] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
        pb.term[g] = (TERM_COLOR << 30) | ((unsigned)depth << TERM_DEPTH_SHIFT) | (unsigned)s;
        qs[s] = -1;
      } else {
        // WShadingPoint::create_rays, hitable.rs:42-47
        const f3 no = sp.point + sp.normal * dm::signum(dot(sp.normal, se.wi)) * sp.offset_by;
        if (!any_nan(new_throughput)) throughput = new_throughput;  // :181-183
        pb.o_time[g] = make_float4(no.x, no.y, no.z, sp.time);
        pb.d_t[g] = make_float4(se.wi.x, se.wi.y, se.wi.z, 0.0f);
        pb.rad[g] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
        pb.thr[g] = make_float4(throughput.x, throughput.y, throughput.z, 0.0f);
      }
    } else {  // :189-203
      pb.rad[g] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
      pb.term[g] = ((depth == 0 ? TERM_BACKGROUND : TERM_COLOR) << 30) | ((unsigned)depth << TERM_DEPTH_SHIFT) | (unsigned)s;
      qs[s] = -1;
    }
  }
  warp_add(pb.counters + CNT_EVALS_SHADOW, evals);
  warp_add(pb.counters + CNT_SHADOW_RAYS, shadows);
}


}  // namespace rt
