// Occupancy-grid sampler + packed (variable samples per ray) compositing: the reference's REAL
// sampling path (SURVEY.md §8 rows a7/a9, "next" row f1).  The reference calls nerfacc 0.5.3
//   estimator.sampling(rays_o, rays_d, sigma_fn=, render_step_size=5e-3, stratified=train,
//                      near_plane=0.0, far_plane=1e10)          src/render/rendering.py:66-74
//   rendering(t_starts, t_ends, ray_indices, n_rays, rgb_sigma_fn, render_bkgd)  :89-96
//   estimator.update_every_n_steps(step, occ_eval_fn, occ_thre=1e-2)   src/run-nerf.py:288-295
// nerfacc's source is not on the box; the semantics implemented here are stated in
// oracle/occgrid.py (parity unpinned against nerfacc itself):
//  * marching: fixed-step intervals [t_k, t_k + dt), t_k = t_begin + k dt with
//    t_begin = max(near plane (+ jitter), entry into the outermost level's box); interval k is
//    emitted iff its midpoint is before min(far plane, exit) and lies in an occupied cell of the
//    finest level whose box contains it.  Two passes (count, exclusive scan by the caller, fill)
//    give ray-major packed output: ray_indices i64 [N], t_starts / t_ends f32 [N].
//  * packed compositing: the dense kernels' arithmetic (composite.cu) on per-ray segments
//    [offsets[r], offsets[r+1]); forward also returns per-sample transmittance, which the
//    backward reads back instead of keeping per-block carries.
//  * grid update: occs[cell] = max(decay * occs[cell], occ); binaries = occs > threshold.
// One warp per ray, lane-strided coalesced accesses, shuffle scans with a running carry.
#include "common.cuh"
#include "../../include/fsnerf_b200.h"

namespace {

constexpr float kEpsF32 = 1.1920928955078125e-07f;
constexpr int kWarps = 8;

__device__ __forceinline__ float warp_incl_scan_add(float v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    float up = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += up;
  }
  return v;
}
__device__ __forceinline__ float warp_suffix_scan_add(float v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    float dn = __shfl_down_sync(0xffffffffu, v, d);
    if (lane + d < 32) v += dn;
  }
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

struct MarchArgs {
  int64_t n_rays;
  const float* rays_o;
  const float* rays_d;
  const float* near_planes;  // [n_rays] (already jittered) or NULL -> near
  float near, far, step;
  const float* aabbs;        // [levels][6] (min xyz, max xyz), level l encloses level l-1
  int levels, res;
  const uint8_t* binaries;   // [levels][res][res][res], z fastest
  const int64_t* offsets;    // [n_rays] exclusive scan of counts (fill pass) or NULL (count pass)
  int32_t* counts;           // [n_rays] (count pass)
  int64_t* ray_indices;
  float* t_starts;
  float* t_ends;
};

// occupancy of point p at the finest level containing it
__device__ __forceinline__ bool occupied(const MarchArgs& a, float px, float py, float pz) {
  for (int l = 0; l < a.levels; ++l) {
    const float* b = a.aabbs + 6 * l;
    if (px >= b[0] && py >= b[1] && pz >= b[2] && px <= b[3] && py <= b[4] && pz <= b[5]) {
      const float fx = (px - b[0]) / (b[3] - b[0]) * (float)a.res;
      const float fy = (py - b[1]) / (b[4] - b[1]) * (float)a.res;
      const float fz = (pz - b[2]) / (b[5] - b[2]) * (float)a.res;
      const int ix = min(max((int)floorf(fx), 0), a.res - 1);
      const int iy = min(max((int)floorf(fy), 0), a.res - 1);
      const int iz = min(max((int)floorf(fz), 0), a.res - 1);
      return a.binaries[(((size_t)l * a.res + ix) * a.res + iy) * a.res + iz] != 0;
    }
  }
  return false;
}

__global__ void __launch_bounds__(kWarps * 32) occgrid_march_kernel(const MarchArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (r >= a.n_rays) return;
  const float ox = a.rays_o[3 * r], oy = a.rays_o[3 * r + 1], oz = a.rays_o[3 * r + 2];
  const float dx = a.rays_d[3 * r], dy = a.rays_d[3 * r + 1], dz = a.rays_d[3 * r + 2];
  // slab test against the outermost level's box
  const float* b = a.aabbs + 6 * (a.levels - 1);
  float t0 = -INFINITY, t1 = INFINITY;
  const float o[3] = {ox, oy, oz}, d[3] = {dx, dy, dz};
  bool miss = false;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if (d[k] != 0.f) {
      const float inv = 1.0f / d[k];
      const float ta = (b[k] - o[k]) * inv, tb = (b[3 + k] - o[k]) * inv;
      t0 = fmaxf(t0, fminf(ta, tb));
      t1 = fminf(t1, fmaxf(ta, tb));
    } else if (o[k] < b[k] || o[k] > b[3 + k]) {
      miss = true;
    }
  }
  const float near = a.near_planes ? a.near_planes[r] : a.near;
  // The samples lie on the lattice near + k * step anchored at the ray's OWN near plane (which
  // carries the stratified jitter): a ray that meets the box behind its near plane starts at the
  // first lattice point at or after the entry, so the jitter survives for cameras outside the box.
  const float t_begin = fmaf(ceilf(fmaxf(t0 - near, 0.f) / a.step), a.step, near), t_limit = fminf(a.far, t1);
  int total = 0;
  const int64_t base = a.offsets ? a.offsets[r] : 0;
  if (!miss && t_limit > t_begin) {
    // candidate k is alive while its midpoint is before the limit: k < (t_limit - t_begin)/dt - 1/2
    const int n_cand = (int)fminf(ceilf((t_limit - t_begin) / a.step), 1.0e7f);
    for (int k0 = 0; k0 < n_cand; k0 += 32) {
      const int k = k0 + lane;
      const float ts = fmaf((float)k, a.step, t_begin);
      const float tm = ts + 0.5f * a.step;
      bool keep = k < n_cand && tm < t_limit;
      if (keep) keep = occupied(a, fmaf(dx, tm, ox), fmaf(dy, tm, oy), fmaf(dz, tm, oz));
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      if (a.offsets && keep) {
        const int64_t p = base + total + __popc(m & ((1u << lane) - 1u));
        a.ray_indices[p] = r;
        a.t_starts[p] = ts;
        a.t_ends[p] = ts + a.step;
      }
      total += __popc(m);
    }
  }
  if (!a.offsets && lane == 0) a.counts[r] = total;
}

// ------------------------------------------------------------------ packed compositing
// One 32-sample block of a ray: the lane's optical depth sd = sigma * delta, alpha = 1 - exp(-sd)
// and transmittance T = exp(-(optical depth of every earlier sample of the ray)).  carry holds the
// ray's optical depth before the block and advances past it.  Lanes past the end pass sigma = 0 and
// t0 = t1 = 0.  The compositing forward and the visibility filter both call this, so the filter
// thresholds exactly the T / alpha the compositor reports.
__device__ __forceinline__ void packed_block_trans(float sigma, float t0, float t1, int lane, float& carry,
                                                   float& alpha, float& T) {
  const float sd = sigma * (t1 - t0);
  alpha = 1.0f - expf(-sd);
  const float incl = warp_incl_scan_add(sd, lane);
  T = expf(-(carry + (incl - sd)));
  carry += __shfl_sync(0xffffffffu, incl, 31);
}

__global__ void __launch_bounds__(kWarps * 32)
composite_packed_fwd_kernel(int64_t n_rays, const int64_t* __restrict__ offsets, const float4* __restrict__ raw,
                            const float* __restrict__ ts, const float* __restrict__ te,
                            const float* __restrict__ bkgd, float* __restrict__ rgb, float* __restrict__ opacity,
                            float* __restrict__ depth, float* __restrict__ weights, float* __restrict__ trans,
                            float* __restrict__ alphas) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (r >= n_rays) return;
  const int64_t base = offsets[r];
  const int S = (int)(offsets[r + 1] - base);
  float acc_r = 0.f, acc_g = 0.f, acc_b = 0.f, acc_w = 0.f, acc_d = 0.f, carry = 0.f;
  for (int s0 = 0; s0 < S; s0 += 32) {
    const int s = s0 + lane;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    float t0 = 0.f, t1 = 0.f;
    if (s < S) {
      c = __ldg(raw + base + s);
      t0 = __ldg(ts + base + s);
      t1 = __ldg(te + base + s);
    }
    float alpha, T;
    packed_block_trans(c.w, t0, t1, lane, carry, alpha, T);
    const float w = T * alpha;
    if (s < S) {
      weights[base + s] = w;
      if (trans) trans[base + s] = T;
      if (alphas) alphas[base + s] = alpha;
      acc_r += w * c.x; acc_g += w * c.y; acc_b += w * c.z;
      acc_w += w;
      acc_d += w * ((t0 + t1) * 0.5f);
    }
  }
  acc_r = warp_sum(acc_r); acc_g = warp_sum(acc_g); acc_b = warp_sum(acc_b);
  acc_w = warp_sum(acc_w); acc_d = warp_sum(acc_d);
  if (lane == 0) {
    acc_d = acc_d / fmaxf(acc_w, kEpsF32);
    if (bkgd) {
      const float om = 1.0f - acc_w;
      acc_r += bkgd[0] * om; acc_g += bkgd[1] * om; acc_b += bkgd[2] * om;
    }
    rgb[r * 3] = acc_r; rgb[r * 3 + 1] = acc_g; rgb[r * 3 + 2] = acc_b;
    opacity[r] = acc_w;
    depth[r] = acc_d;
  }
}

// Visibility filter of OccGridEstimator.sampling (nerfacc's transmittance test): sample i of a ray
// is kept iff T_i >= early_stop_eps and, when alpha_thre > 0, alpha_i >= alpha_thre.  sigma is the
// raw density head and may be negative, so T can rise again along a ray: the kept set is not a
// prefix, and each block is compacted by ballot.  Count pass (out_offsets NULL) writes counts[r];
// the fill pass writes the survivors in their original order from out_offsets[r] on.
__global__ void __launch_bounds__(kWarps * 32)
occgrid_filter_kernel(int64_t n_rays, const int64_t* __restrict__ offsets, const float* __restrict__ ts,
                      const float* __restrict__ te, const float* __restrict__ sigmas, float early_stop_eps,
                      float alpha_thre, const int64_t* __restrict__ out_offsets, int32_t* __restrict__ counts,
                      int64_t* __restrict__ ray_indices, float* __restrict__ ts_out, float* __restrict__ te_out) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (r >= n_rays) return;
  const int64_t base = offsets[r];
  const int S = (int)(offsets[r + 1] - base);
  const int64_t out_base = out_offsets ? out_offsets[r] : 0;
  float carry = 0.f;
  int total = 0;
  for (int s0 = 0; s0 < S; s0 += 32) {
    const int s = s0 + lane;
    float sigma = 0.f, t0 = 0.f, t1 = 0.f;
    if (s < S) {
      sigma = __ldg(sigmas + base + s);
      t0 = __ldg(ts + base + s);
      t1 = __ldg(te + base + s);
    }
    float alpha, T;
    packed_block_trans(sigma, t0, t1, lane, carry, alpha, T);
    const bool keep = s < S && T >= early_stop_eps && (alpha_thre <= 0.f || alpha >= alpha_thre);
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (out_offsets && keep) {
      const int64_t p = out_base + total + __popc(m & ((1u << lane) - 1u));
      ray_indices[p] = r;
      ts_out[p] = t0;
      te_out[p] = t1;
    }
    total += __popc(m);
  }
  if (!out_offsets && lane == 0) counts[r] = total;
}

// x[i] = o[r] + ((d[r] * (t_starts[i] + t_ends[i])) / 2), r = ray_indices[i]: the operation order of
// the drop-in's torch expression (src/render/rendering.py:58-84), rounded op by op with no FMA
// contraction, so x is bit-identical to it.  (torch divides by a scalar through its reciprocal;
// * 0.5 and / 2 round identically.)
__global__ void packed_points_kernel(int64_t n, const int64_t* __restrict__ ray_indices,
                                     const float* __restrict__ ts, const float* __restrict__ te,
                                     const float* __restrict__ rays_o, const float* __restrict__ rays_d,
                                     float* __restrict__ x, float* __restrict__ dirs) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t r = ray_indices[i];
  const float sum = __fadd_rn(__ldg(ts + i), __ldg(te + i));
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float d = __ldg(rays_d + 3 * r + k);
    x[3 * i + k] = __fadd_rn(__ldg(rays_o + 3 * r + k), __fmul_rn(__fmul_rn(d, sum), 0.5f));
    if (dirs) dirs[3 * i + k] = d;
  }
}

// backward: g_i = dL/dw_i = d_rgb.c_i + dA + dDn*m_i (+ d_weights_i);
// dL/d(sigma_i delta_i) = g_i T_{i+1} - sum_{j>i} g_j w_j   (T_{i+1} = T_i - w_i)
__global__ void __launch_bounds__(kWarps * 32)
composite_packed_bwd_kernel(int64_t n_rays, const int64_t* __restrict__ offsets, const float4* __restrict__ raw,
                            const float* __restrict__ ts, const float* __restrict__ te,
                            const float* __restrict__ trans, const float* __restrict__ bkgd,
                            const float* __restrict__ d_rgb, const float* __restrict__ d_opacity,
                            const float* __restrict__ d_depth, const float* __restrict__ d_weights,
                            float4* __restrict__ d_raw, float* __restrict__ d_bkgd) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (r >= n_rays) return;
  const int64_t base = offsets[r];
  const int S = (int)(offsets[r + 1] - base);
  // pass A: opacity and un-normalised depth of the ray (weights from the stored transmittance)
  float acc_w = 0.f, acc_d = 0.f;
  for (int s0 = 0; s0 < S; s0 += 32) {
    const int s = s0 + lane;
    if (s < S) {
      const float t0 = __ldg(ts + base + s), t1 = __ldg(te + base + s);
      const float w = __ldg(trans + base + s) * (1.0f - expf(-__ldg(reinterpret_cast<const float*>(raw + base + s) + 3) * (t1 - t0)));
      acc_w += w;
      acc_d += w * ((t0 + t1) * 0.5f);
    }
  }
  acc_w = warp_sum(acc_w);
  acc_d = warp_sum(acc_d);
  const float gr = d_rgb[r * 3], gg = d_rgb[r * 3 + 1], gb = d_rgb[r * 3 + 2];
  const float gA = d_opacity ? d_opacity[r] : 0.f;
  const float gD = d_depth ? d_depth[r] : 0.f;
  const float den = fmaxf(acc_w, kEpsF32);
  float dA = gA, dDn = gD / den;
  if (acc_w > kEpsF32) dA -= gD * acc_d / (den * den);
  if (bkgd) {
    dA -= gr * bkgd[0] + gg * bkgd[1] + gb * bkgd[2];
    if (d_bkgd && lane == 0) {
      const float om = 1.0f - acc_w;
      atomicAdd(d_bkgd + 0, gr * om);
      atomicAdd(d_bkgd + 1, gg * om);
      atomicAdd(d_bkgd + 2, gb * om);
    }
  }
  // pass B: blocks from the far end of the ray
  float suffix_carry = 0.f;
  for (int s0 = ((S - 1) / 32) * 32; s0 >= 0; s0 -= 32) {
    const int s = s0 + lane;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    float delta = 0.f, tmid = 0.f, T = 0.f, dwv = 0.f;
    if (s < S) {
      c = __ldg(raw + base + s);
      const float t0 = __ldg(ts + base + s), t1 = __ldg(te + base + s);
      delta = t1 - t0;
      tmid = (t0 + t1) * 0.5f;
      T = __ldg(trans + base + s);
      if (d_weights) dwv = __ldg(d_weights + base + s);
    }
    const float w = T * (1.0f - expf(-c.w * delta));
    const float g = gr * c.x + gg * c.y + gb * c.z + dA + dDn * tmid + dwv;
    const float gw = (s < S) ? g * w : 0.f;
    const float incl = warp_suffix_scan_add(gw, lane);
    const float later = suffix_carry + (incl - gw);
    suffix_carry += __shfl_sync(0xffffffffu, incl, 0);
    const float dsd = g * (T - w) - later;
    if (s < S) d_raw[base + s] = make_float4(w * gr, w * gg, w * gb, dsd * delta);
  }
}

// ------------------------------------------------------------------ grid update
// occs[c] = max(decay * occs[c], max over the candidates i that fall in cell c of occ[i]).
// Candidates may share a cell (random subset after warm-up), so the update runs in three
// order-independent phases: gather old values, write decay*old (duplicates write the same
// value), atomic max of the non-negative candidates (signed-int atomicMax on the bit pattern
// is monotone for non-negative floats; a negative candidate never beats decay*old >= 0).
__global__ void occgrid_update_kernel(int phase, int64_t n, const int64_t* __restrict__ cell_ids,
                                      const float* __restrict__ occ, float decay, float* __restrict__ occs,
                                      float* __restrict__ old) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t c = cell_ids ? cell_ids[i] : i;
  if (phase == 0) old[i] = occs[c];
  else if (phase == 1) occs[c] = old[i] * decay;
  else if (occ[i] > 0.f) atomicMax(reinterpret_cast<int*>(occs + c), __float_as_int(occ[i]));
}
__global__ void occgrid_binarize_kernel(int64_t n, const float* __restrict__ occs, float thre,
                                        uint8_t* __restrict__ binaries) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) binaries[i] = occs[i] > thre ? 1 : 0;
}

}  // namespace

extern "C" int fsnerf_occgrid_march(int64_t n_rays, const float* rays_o, const float* rays_d,
                                    const float* near_planes, float near, float far, float step,
                                    const float* aabbs, int levels, int res, const uint8_t* binaries,
                                    const int64_t* offsets, int32_t* counts, int64_t* ray_indices,
                                    float* t_starts, float* t_ends, void* stream) {
  if (n_rays == 0) return FSNERF_OK;
  FS_REQUIRE(rays_o && rays_d && aabbs && binaries, "occgrid_march: null pointer");
  FS_REQUIRE(levels >= 1 && res >= 1 && step > 0.f, "occgrid_march: bad grid / step");
  FS_REQUIRE((offsets && ray_indices && t_starts && t_ends) || (!offsets && counts),
             "occgrid_march: count pass needs counts; fill pass needs offsets and the three outputs");
  MarchArgs a = {n_rays, rays_o, rays_d, near_planes, near, far, step, aabbs, levels, res, binaries,
                 offsets, counts, ray_indices, t_starts, t_ends};
  FsProfScope prof_("occgrid_march", stream);
  occgrid_march_kernel<<<(unsigned)((n_rays + kWarps - 1) / kWarps), kWarps * 32, 0, (cudaStream_t)stream>>>(a);
  return fsnerf_check_launch("occgrid_march");
}

extern "C" int fsnerf_occgrid_filter(int64_t n_rays, const int64_t* offsets, const float* t_starts,
                                     const float* t_ends, const float* sigmas, float early_stop_eps,
                                     float alpha_thre, const int64_t* out_offsets, int32_t* counts,
                                     int64_t* ray_indices, float* out_t_starts, float* out_t_ends, void* stream) {
  if (n_rays == 0) return FSNERF_OK;
  FS_REQUIRE(n_rays > 0 && offsets, "occgrid_filter: bad n_rays / null offsets");
  FS_REQUIRE((out_offsets && ray_indices && out_t_starts && out_t_ends) || (!out_offsets && counts),
             "occgrid_filter: count pass needs counts; fill pass needs out_offsets and the three outputs");
  FsProfScope prof_("occgrid_filter", stream);
  occgrid_filter_kernel<<<(unsigned)((n_rays + kWarps - 1) / kWarps), kWarps * 32, 0, (cudaStream_t)stream>>>(
      n_rays, offsets, t_starts, t_ends, sigmas, early_stop_eps, alpha_thre, out_offsets, counts, ray_indices,
      out_t_starts, out_t_ends);
  return fsnerf_check_launch("occgrid_filter");
}

extern "C" int fsnerf_packed_points(int64_t n, const int64_t* ray_indices, const float* t_starts,
                                    const float* t_ends, const float* rays_o, const float* rays_d, float* x,
                                    float* dirs, void* stream) {
  if (n == 0) return FSNERF_OK;
  FS_REQUIRE(n > 0 && ray_indices && t_starts && t_ends && rays_o && rays_d && x, "packed_points: null pointer");
  FsProfScope prof_("packed_points", stream);
  packed_points_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, ray_indices, t_starts,
                                                                                       t_ends, rays_o, rays_d, x, dirs);
  return fsnerf_check_launch("packed_points");
}

extern "C" int fsnerf_composite_packed_forward(int64_t n_rays, const int64_t* offsets, const float* raw,
                                               const float* t_starts, const float* t_ends, const float* bkgd,
                                               float* rgb, float* opacity, float* depth, float* weights,
                                               float* trans, float* alphas, void* stream) {
  if (n_rays == 0) return FSNERF_OK;
  FS_REQUIRE(offsets && rgb && opacity && depth, "composite_packed_forward: null pointer");
  FS_REQUIRE((reinterpret_cast<uintptr_t>(raw) & 15) == 0, "composite_packed_forward: raw must be 16B aligned");
  FsProfScope prof_("composite_packed_fwd", stream);
  composite_packed_fwd_kernel<<<(unsigned)((n_rays + kWarps - 1) / kWarps), kWarps * 32, 0, (cudaStream_t)stream>>>(
      n_rays, offsets, reinterpret_cast<const float4*>(raw), t_starts, t_ends, bkgd, rgb, opacity, depth, weights,
      trans, alphas);
  return fsnerf_check_launch("composite_packed_forward");
}

extern "C" int fsnerf_composite_packed_backward(int64_t n_rays, const int64_t* offsets, const float* raw,
                                                const float* t_starts, const float* t_ends, const float* trans,
                                                const float* bkgd, const float* d_rgb, const float* d_opacity,
                                                const float* d_depth, const float* d_weights, float* d_raw,
                                                float* d_bkgd, void* stream) {
  if (n_rays == 0) return FSNERF_OK;
  FS_REQUIRE(offsets && d_rgb, "composite_packed_backward: null pointer");
  FS_REQUIRE(((reinterpret_cast<uintptr_t>(raw) | reinterpret_cast<uintptr_t>(d_raw)) & 15) == 0,
             "composite_packed_backward: raw/d_raw must be 16B aligned");
  FsProfScope prof_("composite_packed_bwd", stream);
  composite_packed_bwd_kernel<<<(unsigned)((n_rays + kWarps - 1) / kWarps), kWarps * 32, 0, (cudaStream_t)stream>>>(
      n_rays, offsets, reinterpret_cast<const float4*>(raw), t_starts, t_ends, trans, bkgd, d_rgb, d_opacity,
      d_depth, d_weights, reinterpret_cast<float4*>(d_raw), d_bkgd);
  return fsnerf_check_launch("composite_packed_backward");
}

extern "C" int fsnerf_occgrid_update(int64_t n, const int64_t* cell_ids, const float* occ, float decay,
                                     float* occs, float* workspace, void* stream) {
  if (n == 0) return FSNERF_OK;
  FS_REQUIRE(occ && occs && workspace, "occgrid_update: null pointer (workspace = n floats)");
  FsProfScope prof_("occgrid_update", stream);
  for (int phase = 0; phase < 3; ++phase)
    occgrid_update_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(phase, n, cell_ids, occ,
                                                                                        decay, occs, workspace);
  return fsnerf_check_launch("occgrid_update");
}

extern "C" int fsnerf_occgrid_binarize(int64_t n_cells, const float* occs, float threshold, uint8_t* binaries,
                                       void* stream) {
  if (n_cells == 0) return FSNERF_OK;
  FS_REQUIRE(occs && binaries, "occgrid_binarize: null pointer");
  FsProfScope prof_("occgrid_binarize", stream);
  occgrid_binarize_kernel<<<(unsigned)((n_cells + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n_cells, occs, threshold,
                                                                                             binaries);
  return fsnerf_check_launch("occgrid_binarize");
}
