// C-ABI plumbing (error reporting, device check) + the train-step arithmetic
// kernels (MSE gradient seed, fused Adam) of src/run-nerf.py:216-217,255-258,282-285.
#include <stdarg.h>
#include <stdio.h>
#include "common.cuh"
#include "../../include/fsnerf_b200.h"

static thread_local char g_err[512] = "";

void fsnerf_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int fsnerf_check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    fsnerf_set_error("%s: CUDA launch failed: %s", what, cudaGetErrorString(e));
    return FSNERF_ERR_CUDA;
  }
  return FSNERF_OK;
}

// ---------------------------------------------------------------- profiling
#include <string.h>
#include <vector>
namespace {
struct ProfRec { const char* name; cudaEvent_t a, b; };
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
}  // namespace

FsProfScope::FsProfScope(const char* name, void* st) : slot(-1), stream(st) {
  if (!g_prof_on) return;
  ProfRec r;
  r.name = name;
  if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
  cudaEventRecord(r.a, (cudaStream_t)st);
  g_prof.push_back(r);
  slot = (int)g_prof.size() - 1;
}
FsProfScope::~FsProfScope() {
  if (slot >= 0) cudaEventRecord(g_prof[slot].b, (cudaStream_t)stream);
}

extern "C" int fsnerf_profile_enable(int on) {
  for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_prof.clear();
  g_prof_on = on != 0;
  return FSNERF_OK;
}

extern "C" int fsnerf_profile_read(int max_kernels, char* names, float* total_ms, int* counts) {
  FS_REQUIRE(names && total_ms && counts && max_kernels > 0, "profile_read: null pointer");
  int n = 0;
  for (auto& r : g_prof) {
    if (cudaEventSynchronize(r.b) != cudaSuccess) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
    int k = 0;
    for (; k < n; ++k) if (strncmp(names + 32 * k, r.name, 31) == 0) break;
    if (k == n) {
      if (n == max_kernels) continue;
      strncpy(names + 32 * n, r.name, 31);
      names[32 * n + 31] = 0;
      total_ms[n] = 0.f; counts[n] = 0;
      ++n;
    }
    total_ms[k] += ms;
    counts[k] += 1;
  }
  return n;
}

static void* g_trace = nullptr;
void* fsnerf_debug_trace_ptr() { return g_trace; }
extern "C" int fsnerf_debug_set_trace(void* buf) {
  g_trace = buf;
  return FSNERF_OK;
}

extern "C" int fsnerf_version(void) { return 100; }
extern "C" const char* fsnerf_last_error(void) { return g_err; }

extern "C" int fsnerf_device_ok(int dev) {
  cudaDeviceProp p;
  cudaError_t e = cudaGetDeviceProperties(&p, dev);
  if (e != cudaSuccess) {
    fsnerf_set_error("device_ok: %s", cudaGetErrorString(e));
    return FSNERF_ERR_CUDA;
  }
  if (p.major != 10) {
    fsnerf_set_error("device_ok: device %d is sm_%d%d, this library is sm_100a only", dev, p.major,
                     p.minor);
    return FSNERF_ERR_UNSUPPORTED;
  }
  return FSNERF_OK;
}

namespace {

__global__ void mse_loss_grad_kernel(int64_t n, const float* __restrict__ rgb,
                                     const float* __restrict__ gt, float grad_scale,
                                     float* __restrict__ loss_sum, float* __restrict__ d_rgb) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float sq = 0.f;
  if (i < n) {
    float d = rgb[i] - gt[i];
    sq = d * d;
    if (d_rgb) d_rgb[i] = grad_scale * 2.0f * d;
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, m);
  __shared__ float part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sq;
  __syncthreads();
  if (threadIdx.x == 0 && loss_sum) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += part[w];
    atomicAdd(loss_sum, s);
  }
}

// torch.optim.Adam (amsgrad=False, weight_decay=0, maximize=False) single-tensor form:
//   m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2
//   p -= (lr / (1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
__global__ void adam_kernel(int64_t n, float* __restrict__ p, const float* __restrict__ g,
                            float* __restrict__ m, float* __restrict__ v, float step_size,
                            float b1, float b2, float eps, float inv_sqrt_bc2) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float gi = g[i];
  float mi = b1 * m[i] + (1.0f - b1) * gi;
  float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
  p[i] = p[i] - step_size * (mi / denom);
}

// Weight-norm ("frequency") regulariser of src/run-nerf.py:266-279 fused into the optimiser:
// loss += alpha * sum_t |W_t|_1 ('l1') or alpha * sum_t ||W_t||_F ('l2') over the weight
// tensors with shape[0] > 3, i.e. grad += alpha*sign(w) or alpha*w/||W_t||_F, applied AFTER the
// data-parallel all-reduce so it is added once, not once per rank.
constexpr int kMaxRegSegs = 32;
struct RegSegs {
  int n, mode;            // mode 1 = l1, 2 = l2 (Frobenius norm per tensor)
  float alpha;
  int64_t begin[kMaxRegSegs], end[kMaxRegSegs];
};

// one block-strided pass per segment: sums[seg] += sum |w| (l1) or sum w^2 (l2)
__global__ void reg_norm_kernel(const __grid_constant__ RegSegs segs, const float* __restrict__ p,
                                float* __restrict__ sums) {
  const int seg = blockIdx.y;
  const int64_t b = segs.begin[seg], e = segs.end[seg];
  float acc = 0.f;
  for (int64_t i = b + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < e;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float w = p[i];
    acc += segs.mode == 1 ? fabsf(w) : w * w;
  }
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, m);
  __shared__ float part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += part[w];
    atomicAdd(sums + seg, s);
  }
}

__global__ void adam_reg_kernel(int64_t n, float* __restrict__ p, const float* __restrict__ g,
                                float* __restrict__ m, float* __restrict__ v, float step_size,
                                float b1, float b2, float eps, float inv_sqrt_bc2,
                                const __grid_constant__ RegSegs segs, const float* __restrict__ sums) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float pi = p[i];
  float gi = g[i];
  for (int s = 0; s < segs.n; ++s) {
    if (i >= segs.begin[s] && i < segs.end[s]) {
      if (segs.mode == 1) {
        gi += segs.alpha * (pi > 0.f ? 1.f : (pi < 0.f ? -1.f : 0.f));  // torch.abs backward: sign(w)
      } else {
        gi += segs.alpha * (pi / sqrtf(sums[s]));  // d sqrt(sum w^2) = w / ||W||_F
      }
      break;
    }
  }
  float mi = b1 * m[i] + (1.0f - b1) * gi;
  float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
  p[i] = pi - step_size * (mi / denom);
}

}  // namespace

extern "C" int fsnerf_mse_loss_grad(int64_t n, const float* rgb, const float* gt, float grad_scale,
                                    float* loss_sum, float* d_rgb, void* stream) {
  FS_REQUIRE(rgb && gt, "mse_loss_grad: null pointer");
  if (n <= 0) return FSNERF_OK;
  int threads = 256;
  FsProfScope prof_("mse_loss_grad", stream);
  mse_loss_grad_kernel<<<(unsigned)((n + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
      n, rgb, gt, grad_scale, loss_sum, d_rgb);
  return fsnerf_check_launch("mse_loss_grad");
}

extern "C" int fsnerf_adam_step(int64_t n, float* params, const float* grads, float* m, float* v,
                                float lr, float beta1, float beta2, float eps, int step,
                                void* stream) {
  FS_REQUIRE(params && grads && m && v, "adam_step: null pointer");
  FS_REQUIRE(step >= 1, "adam_step: step counts from 1");
  if (n <= 0) return FSNERF_OK;
  double bc1 = 1.0 - pow((double)beta1, step), bc2 = 1.0 - pow((double)beta2, step);
  float step_size = (float)((double)lr / bc1);
  float inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  int threads = 256;
  FsProfScope prof_("adam", stream);
  adam_kernel<<<(unsigned)((n + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
      n, params, grads, m, v, step_size, beta1, beta2, eps, inv_sqrt_bc2);
  return fsnerf_check_launch("adam_step");
}

// norm_blocks: blocks per regularised tensor in the norm pass.  16 spread each sum over the GPU;
// 1 gives each sum one fixed order (its block adds once to the zeroed sum), so the update is
// reproducible bit for bit.
static int adam_step_reg_impl(int64_t n, float* params, const float* grads, float* m, float* v, float lr,
                              float beta1, float beta2, float eps, int step, int reg_mode, float reg_alpha,
                              int n_segs, const int64_t* seg_begin, const int64_t* seg_end, float* seg_sums,
                              int norm_blocks, void* stream) {
  FS_REQUIRE(params && grads && m && v, "adam_step_reg: null pointer");
  FS_REQUIRE(step >= 1, "adam_step_reg: step counts from 1");
  FS_REQUIRE(reg_mode == 1 || reg_mode == 2, "adam_step_reg: reg_mode must be 1 (l1) or 2 (l2)");
  FS_REQUIRE(n_segs >= 1 && n_segs <= kMaxRegSegs && seg_begin && seg_end && seg_sums,
             "adam_step_reg: 1..32 regularised tensors and a float[n_segs] workspace required");
  if (n <= 0) return FSNERF_OK;
  RegSegs segs;
  segs.n = n_segs; segs.mode = reg_mode; segs.alpha = reg_alpha;
  for (int s = 0; s < n_segs; ++s) {
    FS_REQUIRE(seg_begin[s] >= 0 && seg_begin[s] < seg_end[s] && seg_end[s] <= n,
               "adam_step_reg: segment out of range");
    segs.begin[s] = seg_begin[s]; segs.end[s] = seg_end[s];
  }
  cudaStream_t st = (cudaStream_t)stream;
  double bc1 = 1.0 - pow((double)beta1, step), bc2 = 1.0 - pow((double)beta2, step);
  float step_size = (float)((double)lr / bc1);
  float inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  int threads = 256;
  FsProfScope prof_("adam", stream);
  // seg_sums doubles as the value of the penalty: sum|w| (l1) or sum w^2 (l2) per tensor
  if (cudaMemsetAsync(seg_sums, 0, sizeof(float) * n_segs, st) != cudaSuccess)
    return fsnerf_check_launch("adam_step_reg(memset)");
  reg_norm_kernel<<<dim3(norm_blocks, n_segs), threads, 0, st>>>(segs, params, seg_sums);
  adam_reg_kernel<<<(unsigned)((n + threads - 1) / threads), threads, 0, st>>>(
      n, params, grads, m, v, step_size, beta1, beta2, eps, inv_sqrt_bc2, segs, seg_sums);
  return fsnerf_check_launch("adam_step_reg");
}

extern "C" int fsnerf_adam_step_reg(int64_t n, float* params, const float* grads, float* m, float* v,
                                    float lr, float beta1, float beta2, float eps, int step,
                                    int reg_mode, float reg_alpha, int n_segs,
                                    const int64_t* seg_begin, const int64_t* seg_end,
                                    float* seg_sums, void* stream) {
  return adam_step_reg_impl(n, params, grads, m, v, lr, beta1, beta2, eps, step, reg_mode, reg_alpha, n_segs,
                            seg_begin, seg_end, seg_sums, 16, stream);
}

extern "C" int fsnerf_adam_step_reg_deterministic(int64_t n, float* params, const float* grads, float* m,
                                                  float* v, float lr, float beta1, float beta2, float eps,
                                                  int step, int reg_mode, float reg_alpha, int n_segs,
                                                  const int64_t* seg_begin, const int64_t* seg_end,
                                                  float* seg_sums, void* stream) {
  return adam_step_reg_impl(n, params, grads, m, v, lr, beta1, beta2, eps, step, reg_mode, reg_alpha, n_segs,
                            seg_begin, seg_end, seg_sums, 1, stream);
}
