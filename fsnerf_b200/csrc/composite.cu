// Kernel (4): alpha compositing forward/backward — a per-ray segmented
// transmittance scan.  HBM-bound: one warp per ray, lane-strided so that every
// global access is a fully coalesced 128 B (t) or 512 B (raw float4) line;
// the prefix (forward) and suffix (backward) scans run in registers with
// warp shuffles and a running carry across 32-sample blocks.
//
// Two ray layouts: dense [R,S] (ray r owns [r*S, r*S+S)) and packed (ray r owns
// [offsets[r], offsets[r+1]), the occupancy-grid sampler's output).  One forward kernel serves
// both.  The packed backward is a kernel of its own: a packed ray has no length bound, so it reads
// the forward's per-sample T back instead of keeping per-block carries.  The occupancy-grid
// visibility filter is the same transmittance with a threshold applied.  All of them take T and
// alpha from block_trans, so the backward recomputes exactly the forward's T and the filter
// thresholds exactly the T / alpha the compositor reports.
//
// Semantics (flags == 0): nerfacc.volrend.rendering v0.5.3 as called at
// /root/reference/src/render/rendering.py:89-96 (SURVEY.md Appendix A5);
// oracle/compositing.py:composite_dense restates it.
#include "common.cuh"
#include "../../include/fsnerf_b200.h"

namespace {

constexpr float kEpsF32 = 1.1920928955078125e-07f;  // torch.finfo(float32).eps
constexpr int kWarpsPerBlock = 8;
// Register blocks of the packed forward.  Measured on a B200 (1000 W power limit): NB 2 takes
// the same time as NB 1 at 0.2-0.7 M samples and 17-22 % less at 3-6 M; NB 4 spills registers.
constexpr int kPackedNB = 2;

__device__ __forceinline__ float warp_incl_scan_add(float v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    float up = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += up;
  }
  return v;
}
__device__ __forceinline__ float warp_incl_scan_mul(float v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    float up = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v *= up;
  }
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}
// suffix (reverse) inclusive scan: lane l gets sum_{k>=l} v_k
__device__ __forceinline__ float warp_suffix_scan_add(float v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    float dn = __shfl_down_sync(0xffffffffu, v, d);
    if (lane + d < 32) v += dn;
  }
  return v;
}

// One 32-sample block of a ray: the lane's optical depth sd = sigma * delta gives
// alpha = 1 - exp(-sd) and the transmittance T over every earlier sample of the ray.  carry holds
// the ray's running state before the block and advances past it.  Lanes past the end pass sd = 0.
//   exp-sum form (the reference):  T_i = exp(-sum_{j<i} sd_j), carry = optical depth (starts at 0)
//   product form (FSNERF_COMP_PRODUCT_TRANS):  T_i = prod_{j<i} (1 - alpha_j + 1e-10), carry =
//   product (starts at 1)
struct BlockTrans { float alpha, T; };
__device__ __forceinline__ BlockTrans block_trans(float sd, bool prod, int lane, float& carry) {
  const float alpha = 1.0f - expf(-sd);
  float T;
  if (!prod) {
    const float incl = warp_incl_scan_add(sd, lane);
    T = expf(-(carry + (incl - sd)));
    carry += __shfl_sync(0xffffffffu, incl, 31);
  } else {
    const float f = 1.0f - alpha + 1e-10f;
    const float incl = warp_incl_scan_mul(f, lane);
    float excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.0f;
    T = carry * excl;
    carry *= __shfl_sync(0xffffffffu, incl, 31);
  }
  return {alpha, T};
}

// Occlusion regulariser of src/core/loss.py:26-60 as called at src/run-nerf.py:260-264, fused
// into the compositing backward: loss = mean_r sum_s w(t_mid) * sigma_raw, so
// d(loss)/d(sigma_raw) = scale * w(t_mid) with scale = 1/(rays in the GLOBAL batch).
// func: 0 off, 1 'linear' w = -a t + b, 2 'exp' w = a exp(-b t).  loss (may be NULL)
// accumulates the UNSCALED sum over this launch's rays.
struct OccReg { int func; float a, b, scale; float* loss; };
__device__ __forceinline__ float occ_weight(const OccReg& o, float t) {
  return o.func == 1 ? fmaf(-o.a, t, o.b) : o.a * expf(-o.b * t);
}

__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float ld_stream_f(const float* p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

// NB = number of 32-sample blocks held in registers at once.  Per-lane sums and the carry advance
// block by block in ascending order whatever NB is, so every NB gives the same bits.
// kPacked: ray r is [offsets[r], offsets[r+1]) and S is ignored; otherwise [r*S, r*S+S) and
// offsets is ignored (it comes last: ahead of the others it would move their offsets and
// alignment, and with them the code compiled for the dense kernels).
template <int NB, bool kPacked>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_fwd_kernel(int64_t n_rays, int S, const float4* __restrict__ raw,
                     const float* __restrict__ ts, const float* __restrict__ te,
                     const float* __restrict__ dscale, const float* __restrict__ bkgd, int flags,
                     float* __restrict__ rgb, float* __restrict__ opacity,
                     float* __restrict__ depth, float* __restrict__ weights,
                     float* __restrict__ alphas, float* __restrict__ trans,
                     const int64_t* __restrict__ offsets) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (r >= n_rays) return;
  const int64_t base = kPacked ? offsets[r] : r * S;
  if (kPacked) S = (int)(offsets[r + 1] - base);
  const float ds = dscale ? dscale[r] : 1.0f;
  const bool relu = flags & FSNERF_COMP_SIGMA_RELU;
  const bool prod = flags & FSNERF_COMP_PRODUCT_TRANS;
  float acc_r = 0.f, acc_g = 0.f, acc_b = 0.f, acc_w = 0.f, acc_d = 0.f;
  float carry = prod ? 1.0f : 0.0f;
  for (int s0 = 0; s0 < S; s0 += 32 * NB) {
    float4 c[NB];
    float t0[NB], t1[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      int s = s0 + b * 32 + lane;
      if (s < S) {
        c[b] = ld_stream_f4(raw + base + s);
        t0[b] = ld_stream_f(ts + base + s);
        t1[b] = ld_stream_f(te + base + s);
      } else {
        c[b] = make_float4(0.f, 0.f, 0.f, 0.f);
        t0[b] = t1[b] = 0.f;
      }
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      int s = s0 + b * 32 + lane;
      if (s0 + b * 32 >= S) break;  // warp-uniform
      float sig = relu ? fmaxf(c[b].w, 0.f) : c[b].w;
      float sd = sig * ((t1[b] - t0[b]) * ds);
      const BlockTrans bt = block_trans(sd, prod, lane, carry);
      float w = bt.T * bt.alpha;
      if (s < S) {
        weights[base + s] = w;
        if (alphas) alphas[base + s] = bt.alpha;
        if (trans) trans[base + s] = bt.T;
        acc_r += w * c[b].x;
        acc_g += w * c[b].y;
        acc_b += w * c[b].z;
        acc_w += w;
        acc_d += w * ((t0[b] + t1[b]) * 0.5f);
      }
    }
  }
  acc_r = warp_sum(acc_r); acc_g = warp_sum(acc_g); acc_b = warp_sum(acc_b);
  acc_w = warp_sum(acc_w); acc_d = warp_sum(acc_d);
  if (lane == 0) {
    if (!(flags & FSNERF_COMP_DEPTH_UNNORM)) acc_d = acc_d / fmaxf(acc_w, kEpsF32);
    if (bkgd) {
      float om = 1.0f - acc_w;
      acc_r += bkgd[0] * om; acc_g += bkgd[1] * om; acc_b += bkgd[2] * om;
    }
    rgb[r * 3 + 0] = acc_r; rgb[r * 3 + 1] = acc_g; rgb[r * 3 + 2] = acc_b;
    opacity[r] = acc_w;
    depth[r] = acc_d;
  }
}

// Backward.  With sd_i = sigma_i*delta_i, w_i = T_i*alpha_i:
//   g_i   = dL/dw_i = d_rgb.c_i + dA + dDn*m_i + d_weights_i
//   exp-sum form:  dL/dsd_i = g_i*T_{i+1} - sum_{j>i} g_j w_j
//   product form:  dL/dsd_i = (1-a_i) * (g_i*T_i - sum_{j>i} g_j w_j / (1-a_i+1e-10))
// dA and dDn are the per-ray terms of the opacity, the (normalised) depth and the background.
struct RayGrad { float gr, gg, gb, dA, dDn; };
// acc_w / acc_d: the ray's opacity and un-normalised depth (warp-reduced).  Adds the ray's share
// of d_bkgd (atomics) when d_bkgd is not NULL.
__device__ __forceinline__ RayGrad ray_grad(int64_t r, int lane, float acc_w, float acc_d, bool depth_unnorm,
                                            const float* __restrict__ d_rgb, const float* __restrict__ d_opacity,
                                            const float* __restrict__ d_depth, const float* __restrict__ bkgd,
                                            float* __restrict__ d_bkgd) {
  const float gr = d_rgb[r * 3], gg = d_rgb[r * 3 + 1], gb = d_rgb[r * 3 + 2];
  const float gA = d_opacity ? d_opacity[r] : 0.f;
  const float gD = d_depth ? d_depth[r] : 0.f;
  float dA = gA, dDn = gD;
  if (!depth_unnorm) {
    const float den = fmaxf(acc_w, kEpsF32);
    dDn = gD / den;
    if (acc_w > kEpsF32) dA -= gD * acc_d / (den * den);
  }
  if (bkgd) {
    const float dot = gr * bkgd[0] + gg * bkgd[1] + gb * bkgd[2];
    dA -= dot;
    if (d_bkgd && lane == 0) {
      const float om = 1.0f - acc_w;
      atomicAdd(d_bkgd + 0, gr * om);
      atomicAdd(d_bkgd + 1, gg * om);
      atomicAdd(d_bkgd + 2, gb * om);
    }
  }
  return {gr, gg, gb, dA, dDn};
}

// One 32-sample block of the backward, walked from the far end of the ray: dL/dsd of the lane's
// sample.  suffix_carry = sum of g_j w_j over the later blocks; it advances past this block.
template <bool kProd>
__device__ __forceinline__ float block_dsd(const RayGrad& q, float4 c, float tmid, float dwv, float alpha,
                                           float T, float w, bool valid, int lane, float& suffix_carry) {
  const float g = q.gr * c.x + q.gg * c.y + q.gb * c.z + q.dA + q.dDn * tmid + dwv;
  const float gw = valid ? g * w : 0.f;
  const float incl = warp_suffix_scan_add(gw, lane);
  const float later = suffix_carry + (incl - gw);  // strictly after s
  suffix_carry += __shfl_sync(0xffffffffu, incl, 0);
  if (kProd) {
    const float om = 1.0f - alpha;
    return om * (g * T - later / (om + 1e-10f));
  }
  return g * (T - w) - later;  // T_{i+1} = T_i (1-alpha_i) = T_i - w_i
}

// Dense backward in two passes over the ray instead of holding it in registers: pass A is the
// forward scan (per-block carry-ins, opacity and depth sums), pass B walks the blocks backwards,
// re-reads them (L1/L2 hits: a ray is 4.6 KB), recomputes T with the forward's block_trans from
// the block's carry-in and runs the suffix scan.  Small register state -> many
// resident warps -> HBM stays busy.  NB = 32-sample blocks per ray (S <= 32*NB).
template <int NB, bool kOcc, bool kProd>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, 4)
composite_bwd_stream_kernel(int64_t n_rays, int S, const float4* __restrict__ raw,
                            const float* __restrict__ ts, const float* __restrict__ te,
                            const float* __restrict__ dscale, const float* __restrict__ bkgd, int flags,
                            const float* __restrict__ d_rgb, const float* __restrict__ d_opacity,
                            const float* __restrict__ d_depth, const float* __restrict__ d_weights,
                            float4* __restrict__ d_raw, float* __restrict__ d_bkgd, const OccReg occ) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (r >= n_rays) return;
  const int64_t base = r * S;
  const float ds = dscale ? dscale[r] : 1.0f;
  const bool relu = flags & FSNERF_COMP_SIGMA_RELU;
  float cin[NB];
  float carry = kProd ? 1.0f : 0.0f, acc_w = 0.f, acc_d = 0.f;
  // ---- pass A: forward scan
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    cin[b] = carry;
    if (b * 32 >= S) continue;  // warp-uniform
    const int s = b * 32 + lane;
    float sd = 0.f, tmid = 0.f;
    if (s < S) {
      const float sigma = __ldg(reinterpret_cast<const float*>(raw + base + s) + 3);
      const float t0 = __ldg(ts + base + s), t1 = __ldg(te + base + s);
      sd = (relu ? fmaxf(sigma, 0.f) : sigma) * ((t1 - t0) * ds);
      tmid = (t0 + t1) * 0.5f;
    }
    const BlockTrans bt = block_trans(sd, kProd, lane, carry);
    const float w = bt.T * (1.0f - expf(-sd));  // = bt.T * bt.alpha, spelt so to keep ptxas's schedule of the exp-sum kernels
    if (s < S) {
      acc_w += w;
      acc_d += w * tmid;
    }
  }
  acc_w = warp_sum(acc_w);
  acc_d = warp_sum(acc_d);
  const RayGrad q = ray_grad(r, lane, acc_w, acc_d, flags & FSNERF_COMP_DEPTH_UNNORM, d_rgb, d_opacity, d_depth,
                             bkgd, d_bkgd);
  // ---- pass B: backward over the blocks
  float suffix_carry = 0.f;  // sum over later blocks of g_j w_j
  float occ_acc = 0.f;
#pragma unroll
  for (int b = NB - 1; b >= 0; --b) {
    if (b * 32 >= S) continue;
    const int s = b * 32 + lane;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    float delta = 0.f, tmid = 0.f, dwv = 0.f;
    if (s < S) {
      c = __ldg(raw + base + s);
      const float t0 = __ldg(ts + base + s), t1 = __ldg(te + base + s);
      delta = (t1 - t0) * ds;
      tmid = (t0 + t1) * 0.5f;
      if (d_weights) dwv = ld_stream_f(d_weights + base + s);
    }
    const float sd = (relu ? fmaxf(c.w, 0.f) : c.w) * delta;
    float block_carry = cin[b];
    const BlockTrans bt = block_trans(sd, kProd, lane, block_carry);
    const float w = bt.T * bt.alpha;
    const float dsd = block_dsd<kProd>(q, c, tmid, dwv, bt.alpha, bt.T, w, s < S, lane, suffix_carry);
    float dsig = dsd * delta;
    if (relu && c.w <= 0.f) dsig = 0.f;
    if (kOcc && s < S) {  // compiled out of the plain kernel: its register count sets the occupancy
      const float ow = occ_weight(occ, tmid);
      dsig = fmaf(occ.scale, ow, dsig);
      occ_acc = fmaf(ow, c.w, occ_acc);
    }
    if (s < S) __stcs(d_raw + base + s, make_float4(w * q.gr, w * q.gg, w * q.gb, dsig));  // write-once stream
  }
  if (kOcc && occ.loss) {
    occ_acc = warp_sum(occ_acc);
    if (lane == 0) atomicAdd(occ.loss, occ_acc);
  }
}

// Packed backward (exp-sum form, flags == 0).  A packed ray has no length bound, so per-block
// carries cannot live in registers: both passes read the forward's per-sample T instead.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_packed_bwd_kernel(int64_t n_rays, const int64_t* __restrict__ offsets, const float4* __restrict__ raw,
                            const float* __restrict__ ts, const float* __restrict__ te,
                            const float* __restrict__ trans, const float* __restrict__ bkgd,
                            const float* __restrict__ d_rgb, const float* __restrict__ d_opacity,
                            const float* __restrict__ d_depth, const float* __restrict__ d_weights,
                            float4* __restrict__ d_raw, float* __restrict__ d_bkgd) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
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
  const RayGrad q = ray_grad(r, lane, acc_w, acc_d, false, d_rgb, d_opacity, d_depth, bkgd, d_bkgd);
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
    const float alpha = 1.0f - expf(-c.w * delta);
    const float w = T * alpha;
    const float dsd = block_dsd<false>(q, c, tmid, dwv, alpha, T, w, s < S, lane, suffix_carry);
    if (s < S) d_raw[base + s] = make_float4(w * q.gr, w * q.gg, w * q.gb, dsd * delta);
  }
}

// Visibility filter of OccGridEstimator.sampling (nerfacc's transmittance test): sample i of a ray
// is kept iff T_i >= early_stop_eps and, when alpha_thre > 0, alpha_i >= alpha_thre.  sigma is the
// raw density head and may be negative, so T can rise again along a ray: the kept set is not a
// prefix, and each block is compacted by ballot.  Count pass (out_offsets NULL) writes counts[r];
// the fill pass writes the survivors in their original order from out_offsets[r] on.
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
occgrid_filter_kernel(int64_t n_rays, const int64_t* __restrict__ offsets, const float* __restrict__ ts,
                      const float* __restrict__ te, const float* __restrict__ sigmas, float early_stop_eps,
                      float alpha_thre, const int64_t* __restrict__ out_offsets, int32_t* __restrict__ counts,
                      int64_t* __restrict__ ray_indices, float* __restrict__ ts_out, float* __restrict__ te_out) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
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
    const BlockTrans bt = block_trans(sigma * (t1 - t0), false, lane, carry);
    const bool keep = s < S && bt.T >= early_stop_eps && (alpha_thre <= 0.f || bt.alpha >= alpha_thre);
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

}  // namespace

extern "C" int fsnerf_composite_forward(int64_t n_rays, int n_samples, const float* raw,
                                        const float* t_starts, const float* t_ends,
                                        const float* delta_scale, const float* bkgd, int flags,
                                        float* rgb, float* opacity, float* depth, float* weights,
                                        float* alphas, float* trans, void* stream) {
  if (n_rays == 0) return FSNERF_OK;
  FS_REQUIRE(raw && t_starts && t_ends && rgb && opacity && depth && weights,
             "composite_forward: null pointer");
  FS_REQUIRE(n_samples >= 1 && n_rays >= 0, "composite_forward: bad sizes");
  FS_REQUIRE((reinterpret_cast<uintptr_t>(raw) & 15) == 0, "composite_forward: raw must be 16B aligned");
  unsigned blocks = (unsigned)((n_rays + kWarpsPerBlock - 1) / kWarpsPerBlock);
  cudaStream_t st = (cudaStream_t)stream;
  const float4* raw4 = reinterpret_cast<const float4*>(raw);
#define LAUNCH(NB)                                                                              \
  composite_fwd_kernel<NB, false><<<blocks, kWarpsPerBlock * 32, 0, st>>>(                      \
      n_rays, n_samples, raw4, t_starts, t_ends, delta_scale, bkgd, flags, rgb, opacity, depth, \
      weights, alphas, trans, nullptr)
  FsProfScope prof_("composite_fwd", stream);
  if (n_samples <= 64) LAUNCH(2);
  else if (n_samples <= 128) LAUNCH(4);
  else if (n_samples <= 192) LAUNCH(6);
  else LAUNCH(8);
#undef LAUNCH
  return fsnerf_check_launch("composite_forward");
}

static int composite_backward_impl(int64_t n_rays, int n_samples, const float* raw,
                                   const float* t_starts, const float* t_ends,
                                   const float* delta_scale, const float* bkgd, int flags,
                                   const float* d_rgb, const float* d_opacity,
                                   const float* d_depth, const float* d_weights, float* d_raw,
                                   float* d_bkgd, const OccReg occ, void* stream);

extern "C" int fsnerf_composite_backward(int64_t n_rays, int n_samples, const float* raw,
                                         const float* t_starts, const float* t_ends,
                                         const float* delta_scale, const float* bkgd, int flags,
                                         const float* d_rgb, const float* d_opacity,
                                         const float* d_depth, const float* d_weights, float* d_raw,
                                         float* d_bkgd, void* stream) {
  const OccReg occ = {0, 0.f, 0.f, 0.f, nullptr};
  return composite_backward_impl(n_rays, n_samples, raw, t_starts, t_ends, delta_scale, bkgd, flags,
                                 d_rgb, d_opacity, d_depth, d_weights, d_raw, d_bkgd, occ, stream);
}

extern "C" int fsnerf_composite_backward_occ(int64_t n_rays, int n_samples, const float* raw,
                                             const float* t_starts, const float* t_ends,
                                             const float* delta_scale, const float* bkgd, int flags,
                                             const float* d_rgb, const float* d_opacity,
                                             const float* d_depth, const float* d_weights,
                                             float* d_raw, float* d_bkgd, int occ_func, float occ_a,
                                             float occ_b, float occ_scale, float* occ_loss_sum,
                                             void* stream) {
  FS_REQUIRE(occ_func >= 0 && occ_func <= 2, "composite_backward_occ: occ_func must be 0 (off), 1 (linear) or 2 (exp)");
  FS_REQUIRE(occ_a >= 0.f && occ_b >= 0.f, "composite_backward_occ: a and b should be non-negative");
  const OccReg occ = {occ_func, occ_a, occ_b, occ_scale, occ_loss_sum};
  return composite_backward_impl(n_rays, n_samples, raw, t_starts, t_ends, delta_scale, bkgd, flags,
                                 d_rgb, d_opacity, d_depth, d_weights, d_raw, d_bkgd, occ, stream);
}

using BwdKernel = decltype(&composite_bwd_stream_kernel<2, false, false>);
template <int NB>
static BwdKernel bwd_kernel(bool occ, bool prod) {
  if (occ) return prod ? composite_bwd_stream_kernel<NB, true, true> : composite_bwd_stream_kernel<NB, true, false>;
  return prod ? composite_bwd_stream_kernel<NB, false, true> : composite_bwd_stream_kernel<NB, false, false>;
}

static int composite_backward_impl(int64_t n_rays, int n_samples, const float* raw,
                                   const float* t_starts, const float* t_ends,
                                   const float* delta_scale, const float* bkgd, int flags,
                                   const float* d_rgb, const float* d_opacity,
                                   const float* d_depth, const float* d_weights, float* d_raw,
                                   float* d_bkgd, const OccReg occ, void* stream) {
  if (n_rays == 0) return FSNERF_OK;
  FS_REQUIRE(raw && t_starts && t_ends && d_rgb && d_raw, "composite_backward: null pointer");
  FS_REQUIRE(n_samples >= 1 && n_samples <= 512, "composite_backward: n_samples must be in [1,512]");
  FS_REQUIRE(((reinterpret_cast<uintptr_t>(raw) | reinterpret_cast<uintptr_t>(d_raw)) & 15) == 0,
             "composite_backward: raw/d_raw must be 16B aligned");
  const bool on = occ.func != 0, prod = flags & FSNERF_COMP_PRODUCT_TRANS;
  const BwdKernel k = n_samples <= 64    ? bwd_kernel<2>(on, prod)
                      : n_samples <= 128 ? bwd_kernel<4>(on, prod)
                      : n_samples <= 192 ? bwd_kernel<6>(on, prod)
                      : n_samples <= 256 ? bwd_kernel<8>(on, prod)
                                         : bwd_kernel<16>(on, prod);
  FsProfScope prof_("composite_bwd", stream);
  k<<<(unsigned)((n_rays + kWarpsPerBlock - 1) / kWarpsPerBlock), kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(
      n_rays, n_samples, reinterpret_cast<const float4*>(raw), t_starts, t_ends, delta_scale, bkgd, flags, d_rgb,
      d_opacity, d_depth, d_weights, reinterpret_cast<float4*>(d_raw), d_bkgd, occ);
  return fsnerf_check_launch("composite_backward");
}

// The packed entry points accept NULL per-sample pointers: when every ray is empty the sample
// tensors are empty and the kernels read none of them.
extern "C" int fsnerf_composite_packed_forward(int64_t n_rays, const int64_t* offsets, const float* raw,
                                               const float* t_starts, const float* t_ends, const float* bkgd,
                                               float* rgb, float* opacity, float* depth, float* weights,
                                               float* trans, float* alphas, void* stream) {
  if (n_rays == 0) return FSNERF_OK;
  FS_REQUIRE(offsets && rgb && opacity && depth, "composite_packed_forward: null pointer");
  FS_REQUIRE((reinterpret_cast<uintptr_t>(raw) & 15) == 0, "composite_packed_forward: raw must be 16B aligned");
  FsProfScope prof_("composite_packed_fwd", stream);
  const unsigned blocks = (unsigned)((n_rays + kWarpsPerBlock - 1) / kWarpsPerBlock);
  composite_fwd_kernel<kPackedNB, true><<<blocks, kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(
      n_rays, 0, reinterpret_cast<const float4*>(raw), t_starts, t_ends, nullptr, bkgd, 0, rgb, opacity, depth,
      weights, alphas, trans, offsets);
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
  composite_packed_bwd_kernel<<<(unsigned)((n_rays + kWarpsPerBlock - 1) / kWarpsPerBlock), kWarpsPerBlock * 32, 0,
                                (cudaStream_t)stream>>>(
      n_rays, offsets, reinterpret_cast<const float4*>(raw), t_starts, t_ends, trans, bkgd, d_rgb, d_opacity,
      d_depth, d_weights, reinterpret_cast<float4*>(d_raw), d_bkgd);
  return fsnerf_check_launch("composite_packed_backward");
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
  occgrid_filter_kernel<<<(unsigned)((n_rays + kWarpsPerBlock - 1) / kWarpsPerBlock), kWarpsPerBlock * 32, 0,
                          (cudaStream_t)stream>>>(n_rays, offsets, t_starts, t_ends, sigmas, early_stop_eps, alpha_thre,
                                                  out_offsets, counts, ray_indices, out_t_starts, out_t_ends);
  return fsnerf_check_launch("occgrid_filter");
}
