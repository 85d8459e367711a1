// Occupancy-grid sampler: the reference's REAL sampling path (SURVEY.md §8 rows a7/a9, "next"
// row f1).  The reference calls nerfacc 0.5.3
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
//  * grid update: occs[cell] = max(decay * occs[cell], occ); binaries = occs > threshold.
// One warp per ray for marching, 32 candidates per ballot.  Packed compositing and the visibility
// filter, which are the compositor's transmittance scan, live in composite.cu.
#include "common.cuh"
#include "../../include/fsnerf_b200.h"

namespace {

constexpr int kWarps = 8;

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
