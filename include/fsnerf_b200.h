/* fsnerf_b200 — C ABI of the B200-native fs-nerf ray-march hot path.
 *
 * The reference (a-lemus96/fs-nerf) has no FFI layer: its "operator API" for
 * this path is a handful of Python call sites.  Each entry point below names
 * the reference interface it replaces (file:line relative to the reference
 * repo).  The Python mirror of those interfaces (fsnerf_b200/render/rendering.py,
 * core/models.py, utils/utilities.py) binds this library with ctypes; see
 * INTEGRATION.md for the stub a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success or a negative code
 * (FSNERF_ERR_*); the message is available from fsnerf_last_error().  The
 * library never allocates caller-visible memory: all pointers are DEVICE
 * pointers owned by the caller (contiguous, fp32 unless stated), sizes are
 * explicit, work is enqueued on `stream` (a cudaStream_t passed as void*).
 * There is no CPU fallback: without an sm_100 device every compute call fails.
 */
#ifndef FSNERF_B200_H
#define FSNERF_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FSNERF_OK 0
#define FSNERF_ERR_ARG -1
#define FSNERF_ERR_CUDA -2
#define FSNERF_ERR_UNSUPPORTED -3

/* compositing flags (default 0 == nerfacc.volrend.rendering semantics as
 * called at src/render/rendering.py:89-96; the others are the canonical
 * raw2outputs switches of SURVEY.md Appendix B3) */
#define FSNERF_COMP_SIGMA_RELU 1     /* sigma = relu(raw sigma)                        */
#define FSNERF_COMP_DEPTH_UNNORM 2   /* depth = sum w*t (no division by opacity)        */
#define FSNERF_COMP_PRODUCT_TRANS 4  /* T_i = prod_{j<i}(1-alpha_j+1e-10)               */

int fsnerf_version(void);
const char* fsnerf_last_error(void);
/* 0 if device `dev` can run the kernels (compute capability 10.x) */
int fsnerf_device_ok(int dev);

/* ---- (1) rays --------------------------------------------------------- */
/* Replaces utils.utilities.get_rays (src/utils/utilities.py:36-82) + the NDC
 * warp utils.utilities.to_ndc (:84-120) + the per-item ray-table fetch of
 * LLFFDataset.__getitem__ (src/nerfdata/datasets/llff.py:92-105).
 * Global pixel id p = view*H*W + h*W + w.  pixel_ids==NULL -> p = first_id+i.
 * poses: [n_views, pose_rows(3|4), 4].  images (optional): [n_views,H,W,3]
 * -> rgb_gt[R,3].  sx = -1/(W/(2f)), sy = -1/(H/(2f)) are only read if ndc. */
int fsnerf_gen_rays(const float* poses, int n_views, int pose_rows, int H, int W, float focal,
                    const int64_t* pixel_ids, int64_t first_id, int64_t n_rays, int ndc,
                    float ndc_near, float ndc_sx, float ndc_sy, const float* images, float* rays_o,
                    float* rays_d, float* rgb_gt, void* stream);
/* utils.utilities.to_ndc on existing rays (src/utils/utilities.py:84-120) */
int fsnerf_to_ndc(const float* rays_o, const float* rays_d, int64_t n_rays, float near, float sx,
                  float sy, float* ndc_o, float* ndc_d, void* stream);

/* Stands in for estimator.sampling (src/render/rendering.py:66-74), replaced
 * per BASELINE.json north_star by stratified sampling (SURVEY.md App. B1).
 * u: [R,S] uniforms in [0,1) or NULL (deterministic).  Outputs [R,S]:
 * t_starts = sorted points z, t_ends = [z[1:], far]. */
int fsnerf_sample_stratified(int64_t n_rays, int n_samples, float near, float far, const float* u,
                             float* t_starts, float* t_ends, void* stream);
/* Hierarchical inverse-CDF resampling (SURVEY.md App. B2, warp-tree CDF order).
 * z_coarse (non-decreasing per ray, as sample_stratified emits it), w_coarse [R,Sc];
 * u [R,Sf] or NULL.  Outputs: samples [R,Sf],
 * inds [R,Sf] int32 (searchsorted right), perm [R,Sc+Sf] int32 (stable sort
 * permutation of cat(z_coarse,samples)), t_starts/t_ends [R,Sc+Sf].
 * samples/inds/perm may be NULL. */
int fsnerf_sample_pdf(int64_t n_rays, int n_coarse, int n_fine, const float* z_coarse,
                      const float* w_coarse, const float* u, float far, float* samples,
                      int32_t* inds, int32_t* perm, float* t_starts, float* t_ends, void* stream);

/* Seeded variants: the uniforms the reference draws with torch.rand (src/render/
 * rendering.py stratified jitter / sample_pdf u) come from a stateless counter-based
 * generator evaluated inside the kernel — element i of the [R,S] (resp. [R,Sf]) grid uses
 * fsnerf_rng_uniform's value i for the same seed — so no uniform buffer is written or read.
 * Results are bit-identical to the explicit-u entry points fed with that stream. */
int fsnerf_sample_stratified_seeded(int64_t n_rays, int n_samples, float near, float far,
                                    uint64_t seed, float* t_starts, float* t_ends, void* stream);
int fsnerf_sample_pdf_seeded(int64_t n_rays, int n_coarse, int n_fine, const float* z_coarse,
                             const float* w_coarse, uint64_t seed, float far, float* samples,
                             int32_t* inds, int32_t* perm, float* t_starts, float* t_ends,
                             void* stream);
/* out[i] = u(seed, i) in [0,1), 24 random bits, i < n (oracle/sampling.py:rng_uniform). */
int fsnerf_rng_uniform(int64_t n, uint64_t seed, float* out, void* stream);

/* ---- (4) compositing -------------------------------------------------- */
/* Replaces nerfacc.volrend.rendering as called at src/render/rendering.py:89-96
 * on a dense layout (S samples per ray).  raw [R,S,4]=(rgb,sigma).
 * delta_scale [R] or NULL; bkgd [3] or NULL.  Outputs rgb[R,3], opacity[R],
 * depth[R], weights[R,S]; alphas/trans [R,S] optional (NULL to skip). */
int fsnerf_composite_forward(int64_t n_rays, int n_samples, const float* raw, const float* t_starts,
                             const float* t_ends, const float* delta_scale, const float* bkgd,
                             int flags, float* rgb, float* opacity, float* depth, float* weights,
                             float* alphas, float* trans, void* stream);
/* Backward of the above (the autograd edge of loss.backward(),
 * src/run-nerf.py:282).  d_weights [R,S] or NULL.  Outputs d_raw [R,S,4];
 * d_bkgd [3] (accumulated with atomics, may be NULL). */
int fsnerf_composite_backward(int64_t n_rays, int n_samples, const float* raw,
                              const float* t_starts, const float* t_ends, const float* delta_scale,
                              const float* bkgd, int flags, const float* d_rgb,
                              const float* d_opacity, const float* d_depth, const float* d_weights,
                              float* d_raw, float* d_bkgd, void* stream);

/* Same as fsnerf_composite_backward with the occlusion regulariser
 * (core.loss.OcclusionRegularizer, src/core/loss.py:26-60, added to the loss at
 * src/run-nerf.py:260-264) fused in:  loss_occ = mean_r sum_s w(t_mid)*sigma_raw,
 * w = -a t + b (occ_func 1, 'linear') or a exp(-b t) (occ_func 2, 'exp');
 * d_raw.sigma += occ_scale * w(t_mid)   (occ_scale = 1 / rays of the GLOBAL batch),
 * *occ_loss_sum += sum_r sum_s w*sigma_raw (unscaled; NULL to skip).  occ_func 0 = off. */
int fsnerf_composite_backward_occ(int64_t n_rays, int n_samples, const float* raw,
                                  const float* t_starts, const float* t_ends,
                                  const float* delta_scale, const float* bkgd, int flags,
                                  const float* d_rgb, const float* d_opacity, const float* d_depth,
                                  const float* d_weights, float* d_raw, float* d_bkgd, int occ_func,
                                  float occ_a, float occ_b, float occ_scale, float* occ_loss_sum,
                                  void* stream);

/* ---- (2) standalone positional encoding ---------------------------------- */
/* M.PositionalEncoder.forward (src/core/models.py:43-50): x [P,d_input] ->
 * out [P, d_input*(1+2*n_freqs)] = [x, sin(f_0 x), cos(f_0 x), ...] fp32; freqs
 * [n_freqs] device floats; mask [d_out] (FreeNeRF, Appendix B4) or NULL.  The MLP
 * kernels fuse the same encoding into their first-layer operand staging and never call this. */
int fsnerf_encode(int64_t n_points, int d_input, int n_freqs, const float* freqs, const float* mask,
                  const float* x, float* out, void* stream);

/* ---- occupancy-grid sampler + packed compositing (SURVEY.md §8 f1) -------- */
/* Replaces nerfacc's OccGridEstimator.sampling as called at
 * src/render/rendering.py:66-74 (ray/box slab test + fixed-step marching through
 * binaries[levels][res][res][res], z fastest; aabbs [levels][6], level l encloses l-1).
 * Interval k = [t_begin + k*step, +step), t_begin = the first point of the lattice near + j*step
 * (anchored at the ray's near plane) at or after the box entry; kept iff
 * its midpoint is before min(far, box exit) and in an occupied cell of the finest level
 * containing it.  near_planes [n_rays] (per-ray, jittered when stratified) or NULL -> near.
 * Count pass: offsets == NULL, writes counts[n_rays].  Fill pass: offsets = exclusive scan
 * of counts; writes ray_indices (int64), t_starts, t_ends in ray-major packed order. */
int fsnerf_occgrid_march(int64_t n_rays, const float* rays_o, const float* rays_d,
                         const float* near_planes, float near, float far, float step,
                         const float* aabbs, int levels, int res, const uint8_t* binaries,
                         const int64_t* offsets, int32_t* counts, int64_t* ray_indices,
                         float* t_starts, float* t_ends, void* stream);
/* Visibility filter of OccGridEstimator.sampling (src/render/rendering.py:58-84 passes the
 * density-only sigma_fn; nerfacc's filter keeps a sample iff its transmittance T >= early_stop_eps
 * and, when alpha_thre > 0, alpha >= alpha_thre).  Candidates: ray r owns [offsets[r], offsets[r+1])
 * of t_starts / t_ends / sigmas [N]; T and alpha are bit-identical to
 * fsnerf_composite_packed_forward's trans / alphas of the same sigmas.  sigma may be negative, so
 * the survivors are compacted per ray, not cut at a prefix.  Count pass: out_offsets == NULL,
 * writes counts[n_rays].  Fill pass: out_offsets = exclusive scan of counts; writes the survivors'
 * ray_indices (int64), t_starts, t_ends in their original order. */
int fsnerf_occgrid_filter(int64_t n_rays, const int64_t* offsets, const float* t_starts,
                          const float* t_ends, const float* sigmas, float early_stop_eps, float alpha_thre,
                          const int64_t* out_offsets, int32_t* counts, int64_t* ray_indices,
                          float* out_t_starts, float* out_t_ends, void* stream);
/* Sample points of packed intervals (src/render/rendering.py:58-84):
 * x[i] = rays_o[r] + rays_d[r] * (t_starts[i] + t_ends[i]) / 2 with r = ray_indices[i], rounded in
 * that operation order without FMA contraction; dirs[i] = rays_d[r] when dirs is not NULL. */
int fsnerf_packed_points(int64_t n, const int64_t* ray_indices, const float* t_starts, const float* t_ends,
                         const float* rays_o, const float* rays_d, float* x, float* dirs, void* stream);
/* nerfacc.volrend.rendering (src/render/rendering.py:89-96) on packed samples: ray r owns
 * [offsets[r], offsets[r+1]); raw [N,4] = (rgb, sigma).  Outputs rgb [R,3], opacity [R],
 * depth [R], weights [N]; trans / alphas [N] optional (trans is what the backward reads). */
int fsnerf_composite_packed_forward(int64_t n_rays, const int64_t* offsets, const float* raw,
                                    const float* t_starts, const float* t_ends, const float* bkgd,
                                    float* rgb, float* opacity, float* depth, float* weights,
                                    float* trans, float* alphas, void* stream);
int fsnerf_composite_packed_backward(int64_t n_rays, const int64_t* offsets, const float* raw,
                                     const float* t_starts, const float* t_ends, const float* trans,
                                     const float* bkgd, const float* d_rgb, const float* d_opacity,
                                     const float* d_depth, const float* d_weights, float* d_raw,
                                     float* d_bkgd, void* stream);
/* OccGridEstimator.update_every_n_steps (src/run-nerf.py:288-295): occs[c] = max(decay*occs[c],
 * max of the candidates occ[i] with cell_ids[i] == c) (cell_ids NULL: i == c); workspace n floats.
 * binarize: binaries[c] = occs[c] > threshold. */
int fsnerf_occgrid_update(int64_t n, const int64_t* cell_ids, const float* occ, float decay,
                          float* occs, float* workspace, void* stream);
int fsnerf_occgrid_binarize(int64_t n_cells, const float* occs, float threshold, uint8_t* binaries,
                            void* stream);

/* ---- (2)+(3) NeRF MLP -------------------------------------------------- */
/* Architecture of core.models.NeRF (src/core/models.py:57-109). */
typedef struct fsnerf_net_cfg {
  int n_layers;    /* hidden layers before the bottleneck (8)              */
  int d_hidden;    /* 256 (the tcgen05 path supports 256 only)             */
  int skip_mask;   /* bit i: concat PE(x) after layers[i] (ref skip=[4] -> 16) */
  int n_freqs_pos; /* 10 -> 63 channels                                    */
  int n_freqs_dir; /* 4  -> 27 channels                                    */
  int log_space;   /* 1: f_k = 2^k ; 0: linspace(1, 2^(L-1), L)            */
} fsnerf_net_cfg;

/* Flat fp32 parameter buffer: tensors in the reference's state-dict order
 * (layers.i.weight, layers.i.bias, ..., sigma, connection, branch, rgb;
 * src/core/models.py:96-108), each starting on a 16-byte boundary.
 * fsnerf_mlp_param_count = length of that buffer in floats (incl. padding);
 * fsnerf_mlp_param_layout fills offsets/numels (floats) of every tensor and
 * returns the tensor count (24 for the default net) or a negative code. */
int64_t fsnerf_mlp_param_count(const fsnerf_net_cfg* cfg);
int fsnerf_mlp_param_layout(const fsnerf_net_cfg* cfg, int64_t* offsets, int64_t* numels,
                            int max_tensors);
/* bytes of the packed bf16 operand image (forward + transposed blocks) */
int64_t fsnerf_mlp_packed_bytes(const fsnerf_net_cfg* cfg);
/* bytes of the activation stash the backward needs for n_samples */
int64_t fsnerf_mlp_stash_bytes(const fsnerf_net_cfg* cfg, int64_t n_samples);
/* bytes of scratch the backward needs for n_samples: flow-control flags, the tile table and the
 * ring of d(pre-activation) images that its dgrad CTAs hand to its wgrad CTAs (<= ~100 MB, it does
 * NOT grow with n_samples beyond one launch's worth of CTAs).  Reusing one workspace for every
 * call keeps the ring L2 resident. */
int64_t fsnerf_mlp_bwd_workspace_bytes(const fsnerf_net_cfg* cfg, int64_t n_samples);
/* fp32 params -> packed bf16 SWIZZLE_128B operand blocks */
int fsnerf_mlp_pack(const fsnerf_net_cfg* cfg, const float* params, void* packed, void* stream);

/* Replaces NeRF.forward (src/core/models.py:111-143) evaluated in the closures
 * of render_rays (src/render/rendering.py:58-64,76-84): sample p belongs to ray
 * p / samples_per_ray, position o + d*(t_starts[p]+t_ends[p])/2, view dir d.
 * If x != NULL the positions (and dirs, if given) are read from x/dirs [P,3]
 * instead (plain model(x, dirs) call).  mask_pos [3(1+2Lp)] / mask_dir
 * [3(1+2Ld)] or NULL (FreeNeRF mask, App. B4).  density_only: 0 -> out is [P,4] =
 * (rgb, sigma); 1 -> out is [P] sigma (model(x) form, the view branch is skipped);
 * 2 -> as 1 but sigma is written to the .w slot of a [P,4] buffer (rgb untouched), so a
 * proposal / coarse pass whose colours are not needed feeds the compositor directly.  stash: NULL for inference,
 * else fsnerf_mlp_stash_bytes() bytes kept for the backward. */
int fsnerf_mlp_forward(const fsnerf_net_cfg* cfg, const float* params, const void* packed,
                       int64_t n_samples, int samples_per_ray, const float* rays_o,
                       const float* rays_d, const float* t_starts, const float* t_ends,
                       const float* x, const float* dirs, const float* mask_pos,
                       const float* mask_dir, int density_only, float* out, void* stash,
                       void* stream);
/* Backward of fsnerf_mlp_forward: d_out [P,4] -> grads (fp32, same layout as params;
 * ACCUMULATED into, caller zeroes).  Two launches: the sigma / rgb head weight gradients (SIMT) and
 * ONE persistent cooperative launch (<= 148 CTAs, one per SM) in which dgrad CTAs and wgrad CTAs
 * run side by side and wait on each other through the workspace — the device must be able to
 * hold every CTA of it at once (the launch fails otherwise; nothing else may occupy the GPU).
 * The call resets the workspace flags itself (one small cudaMemsetAsync on `stream`).
 * density_only backward is unsupported (the reference's sigma_fn pass runs under no_grad). */
int fsnerf_mlp_backward(const fsnerf_net_cfg* cfg, const float* params, const void* packed,
                        int64_t n_samples, const void* stash, const float* out,
                        const float* d_out, int density_only, float* grads, void* workspace,
                        void* stream);

/* ---- train-step arithmetic (src/run-nerf.py:216-217,255-258,282-285) ---- */
/* d_rgb = grad_scale*2*(rgb-gt); loss_sum += sum((rgb-gt)^2) (atomic; caller zeroes) */
int fsnerf_mse_loss_grad(int64_t n, const float* rgb, const float* gt, float grad_scale,
                         float* loss_sum, float* d_rgb, void* stream);
/* torch.optim.Adam (defaults) on a flat buffer; step counts from 1 */
int fsnerf_adam_step(int64_t n, float* params, const float* grads, float* m, float* v, float lr,
                     float beta1, float beta2, float eps, int step, void* stream);

/* fsnerf_adam_step with the weight-norm ("frequency") penalty of
 * src/run-nerf.py:266-279 fused in: for every regularised tensor t (flat range
 * [seg_begin[t], seg_end[t]) — the weights with shape[0] > 3)
 *   reg_mode 1 ('l1'): loss += alpha*sum|w|       -> grad += alpha*sign(w)
 *   reg_mode 2 (else): loss += alpha*||W_t||_F    -> grad += alpha*w/||W_t||_F
 * before the Adam update.  seg_sums [n_segs] device floats (workspace AND
 * output): sum|w| (l1) or sum w^2 (l2) per tensor, computed from the
 * PRE-update weights.  n_segs <= 32.  Call it after the data-parallel
 * all-reduce so that the penalty is added once. */
int fsnerf_adam_step_reg(int64_t n, float* params, const float* grads, float* m, float* v, float lr,
                         float beta1, float beta2, float eps, int step, int reg_mode,
                         float reg_alpha, int n_segs, const int64_t* seg_begin,
                         const int64_t* seg_end, float* seg_sums, void* stream);

/* ---- measurement aid (bench.py): per-kernel device time ------------------ */
/* on != 0: start recording a cudaEvent pair around every kernel this library
 * launches (on the launch stream); 0: stop and drop the records. */
int fsnerf_profile_enable(int on);
/* Sum the recorded times by kernel name (synchronises the recorded events).
 * names: max_kernels x 32 chars; returns the number of distinct kernels. */
int fsnerf_profile_read(int max_kernels, char* names, float* total_ms, int* counts);
/* tuning aid: device buffer of >= 2048 int64 that CTA 0 of the MLP forward fills
 * with clock64 phase timestamps (NULL disables; tools/trace_fwd.py decodes it). */
int fsnerf_debug_set_trace(void* buf);

#ifdef __cplusplus
}
#endif
#endif /* FSNERF_B200_H */
