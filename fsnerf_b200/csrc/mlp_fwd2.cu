// Kernels (2)+(3), second generation: the fused NeRF MLP forward with the
// activations resident in TENSOR MEMORY (reference: src/core/models.py:111-143
// evaluated in the closures of src/render/rendering.py:58-84).
//
// One persistent CTA per SM (480 threads), one 128-sample tile at a time:
//   warps 0..7   epilogue: warp w owns TMEM lanes 32*(w&3).. (sample rows) and the
//                column half (w>>2) of every 64-feature chunk.  TMEM -> regs -> bias +
//                ReLU -> bf16x2 -> written back IN PLACE over the fp32 columns just
//                consumed: the next layer's A operand never touches shared memory.
//                Each finished chunk is handed to the MMA warp (mbarrier per chunk), so
//                layer l+1's MMAs on chunk 0 run while chunks 1..3 are still converted.
//   warps 8..11  encoders: ray -> position -> masked sin/cos encoding of position and
//                view direction into two [128 x 64] SW128 smem tiles, one tile ahead.
//   warp 12      MMA issuer: tcgen05.mma M=128 N=256 K=16 kind::f16; A from TMEM
//                (hidden chunks) or smem (encodings), B from the smem weight ring;
//                the two 256-column TMEM regions alternate accumulator / operand role.
//   warps 13..14 weight producers: 32 KB [256 x 64] operand stages L2 -> smem with
//                cp.async.bulk; two issuing warps because bulk copies issued by one
//                thread do not overlap (tools/l2_bench.cu).
// Training (kTrain): every A image (SW128 byte image, the format dgrad / wgrad load
// back) is also staged through smem per 32-row slab and bulk-stored to the stash.
#include "common.cuh"
#include "mlp_common.cuh"
#include "mlp_encode.cuh"
#include "mlp_issue.cuh"

namespace fs {
namespace {

constexpr int kEpiWarps = 8;
constexpr int kEncWarps = 4;
constexpr int kWarpEnc0 = kEpiWarps;               // 8
constexpr int kWarpMma = kEpiWarps + kEncWarps;    // 12, 13
constexpr int kWarpProd0 = kWarpMma + kMmaWarps;   // 14
constexpr int kThreads2 = (kWarpProd0 + kProdWarps) * 32;  // 512
constexpr int kSlabBytes2 = 32 * 128;              // 32 rows of one chunk image
constexpr int kStageBufs = 3;                      // staging buffers per lane quarter
constexpr int kTmemCols2 = 512;
constexpr int kMaxLayers2 = 12;                    // GEMM layers whose biases fit the smem table
static_assert(kMaxHidden + 2 <= kMaxLayers2, "every network build_program accepts must fit the forward");
template <bool kTrain> __host__ __device__ constexpr int n_stages() { return kTrain ? 4 : 5; }
template <bool kTrain> struct Smem {
  static constexpr int ring = 0;
  static constexpr int aux_pos = ring + n_stages<kTrain>() * kStageBytes;
  static constexpr int aux_dir = aux_pos + kChunkBytes;
  static constexpr int staging = aux_dir + kChunkBytes;
  static constexpr int exch = staging + (kTrain ? 4 * kStageBufs * kSlabBytes2 : 0);
  static constexpr int bias = exch + kTileM * 16;              // fp32 [kMaxLayers2][256]
  static constexpr int heads = bias + kMaxLayers2 * 256 * 4;   // fp32 sigma_w[256], rgb_w[3][128]
  static constexpr int bars = heads + 648 * 4;                 // + sigma_b, rgb_b[3] (contiguous in the small block)
  static constexpr int total = bars + 256;
};

// barrier block layout (byte offsets from Smem::bars)
template <bool kTrain> struct Bars {
  static constexpr int S = n_stages<kTrain>();
  static constexpr int w_full = Smem<kTrain>::bars;
  static constexpr int w_empty = w_full + 8 * S;
  static constexpr int a_ready = w_empty + 8 * S;   // [4]
  static constexpr int acc_full = a_ready + 8 * 4;  // [2]
  static constexpr int pos_full = acc_full + 8 * 2;
  static constexpr int pos_empty = pos_full + 8;
  static constexpr int dir_full = pos_empty + 8;
  static constexpr int dir_empty = dir_full + 8;
  static constexpr int token = dir_empty + 8;       // [2] MMA issuers' hand-over
  static constexpr int tmem_slot = token + 16;
  static constexpr int drained = tmem_slot + 8;     // the epilogue has read the tile's last accumulator
};


#define FS_TRACE2(slot, g_, k_)                                                             \
  do {                                                                                      \
    if (args.trace && blockIdx.x == 0 && (slot) < 4)                                        \
      args.trace[((slot) * 16 + (g_)) * 8 + (k_)] = clock64();                              \
  } while (0)

struct Fwd2Args {
  long long* trace;
  const uint8_t* packed;
  int64_t n_samples;
  int samples_per_ray;
  const float* rays_o;
  const float* rays_d;
  const float* t_starts;
  const float* t_ends;
  const float* x;
  const float* dirs;
  const float* mask_pos;
  const float* mask_dir;
  int density_only;
  float* out;
  uint8_t* stash;
};

template <bool kTrain>
__global__ void __launch_bounds__(kThreads2, 1)
mlp_fwd2_kernel(const __grid_constant__ MlpProgram prog, const __grid_constant__ Fwd2Args args,
                const __grid_constant__ IssueTable tab) {
  extern __shared__ __align__(1024) uint8_t smem[];
  using S = Smem<kTrain>;
  constexpr int kStages = n_stages<kTrain>();
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // (shuffle: provably warp-uniform)
  using B = Bars<kTrain>;
  const uint32_t bar_w_full = sbase + B::w_full;       // [kStages]
  const uint32_t bar_w_empty = sbase + B::w_empty;     // [kStages]
  const uint32_t bar_a_ready = sbase + B::a_ready;     // [4]
  const uint32_t bar_acc_full = sbase + B::acc_full;   // [2]
  const uint32_t bar_pos_full = sbase + B::pos_full;
  const uint32_t bar_pos_empty = sbase + B::pos_empty;
  const uint32_t bar_dir_full = sbase + B::dir_full;
  const uint32_t bar_dir_empty = sbase + B::dir_empty;
  const uint32_t bar_token = sbase + B::token;         // [2]
  const uint32_t tmem_slot = sbase + B::tmem_slot;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + B::tmem_slot);
  float4* exch = reinterpret_cast<float4*>(smem + S::exch);

  const int n_gemm = args.density_only ? prog.n_hidden : prog.n_gemm;
  int last_pos_user = 0;  // last hidden layer whose MMA reads the position encoding
  for (int g = 0; g < prog.n_hidden; ++g)
    if (prog.layer[g].use_aux) last_pos_user = g;
  const int64_t n_tiles = (args.n_samples + kTileM - 1) / kTileM;
  const TileSeq seq = TileSeq::strided((int64_t)blockIdx.x, (int64_t)gridDim.x, n_tiles);

  if ((sbase & 1023u) != 0) {
    if (threadIdx.x == 0) printf("fsnerf: dynamic smem base not 1024B aligned (%u)\n", sbase);
    __trap();
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_w_full + 8 * s, 1);
      mbar_init(bar_w_empty + 8 * s, 1);
    }
    for (int c = 0; c < 4; ++c) mbar_init(bar_a_ready + 8 * c, kEpiWarps);
    mbar_init(bar_acc_full, kMmaWarps);
    mbar_init(bar_acc_full + 8, kMmaWarps);
    mbar_init(bar_token, 1);
    mbar_init(bar_token + 8, 1);
    mbar_init(bar_pos_full, kEncWarps);
    mbar_init(bar_pos_empty, 1);
    mbar_init(bar_dir_full, kEncWarps);
    mbar_init(bar_dir_empty, 1);
    mbar_init(sbase + B::drained, kEpiWarps);
    fence_barrier_init();
  }
  if (warp == kWarpMma) {
    tmem_alloc(tmem_slot, kTmemCols2);
    tmem_relinquish();
  }
  // biases: constant bank -> shared memory (the epilogue reads them as broadcast LDS.128;
  // indexed constant loads miss the small constant cache and serialise the epilogue)
  // straight from the packed image's fp32 "small params" block (no per-launch constant upload)
  const float* __restrict__ small = reinterpret_cast<const float*>(args.packed + prog.small_off);
  for (int i = threadIdx.x; i < prog.n_gemm * 256; i += kThreads2)
    reinterpret_cast<float*>(smem + S::bias)[i] = __ldg(small + kSmallBias + i);
  for (int i = threadIdx.x; i < 644; i += kThreads2)  // sigma_w[256], rgb_w[3][128], sigma_b, rgb_b[3]: contiguous
    reinterpret_cast<float*>(smem + S::heads)[i] = __ldg(small + kSmallSigmaW + i);
  const float* head_b = reinterpret_cast<const float*>(smem + S::heads) + 640;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp >= kWarpProd0) {
    // ------------------------------------------------ weight producers
    IssueBars IB{bar_w_full, bar_w_empty, bar_token, sbase + S::ring};
    producer_loop<kStages>(tab, IB, args.packed, seq, warp - kWarpProd0, lane);
  } else if (warp >= kWarpMma) {
    // ------------------------------------------------ MMA issuers (mlp_issue.cuh)
    // Within a layer the encoding chunk (smem operand, independent of the previous epilogue)
    // goes FIRST in the table: it fills the bubble while the epilogue converts chunk 0.
    if (tmem_base != 0) __trap();  // 512 columns = the whole tensor memory
    IssueBars IB{bar_w_full, bar_w_empty, bar_token, sbase + S::ring};
    issuer_loop<kStages>(tab, IB, sbase, seq, (uint32_t)(warp - kWarpMma), lane, args.trace);
  } else if (warp >= kWarpEnc0) {
    // ------------------------------------------------ encoders (thread = sample row)
    const int row = (warp - kWarpEnc0) * 32 + lane;
    uint32_t titer = 0;
    for (int64_t tile; (tile = seq.get(titer)) >= 0; ++titer) {
      const int64_t p = tile * kTileM + row;
      const bool valid = p < args.n_samples;
      float pos[3] = {0.f, 0.f, 0.f}, dir[3] = {0.f, 0.f, 0.f};
      if (valid) {
        if (args.x) {
#pragma unroll
          for (int a = 0; a < 3; ++a) pos[a] = args.x[p * 3 + a];
          if (args.dirs) {
#pragma unroll
            for (int a = 0; a < 3; ++a) dir[a] = args.dirs[p * 3 + a];
          }
        } else {
          const int64_t ray = p / args.samples_per_ray;
          // reference: src/render/rendering.py:79  x = o + d*(ts+te)/2
          const float tm = (args.t_starts[p] + args.t_ends[p]) / 2.0f;
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            dir[a] = args.rays_d[ray * 3 + a];
            pos[a] = args.rays_o[ray * 3 + a] + dir[a] * tm;
          }
        }
      }
      uint8_t* stash_tile = kTrain ? args.stash + (size_t)tile * prog.stash_tile_bytes : nullptr;
      if (kTrain) {  // this warp's previous slab stores must have finished reading the tiles
        if (lane == 0) bulk_wait_read0();
        __syncwarp();
      }
      mbar_wait_relaxed(bar_pos_empty, (titer & 1) ^ 1);
      encode_row(pos, prog.n_freqs_pos, prog.freq_pos, prog.pow2_freqs != 0, args.mask_pos,
                 sbase + S::aux_pos, row);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_pos_full);
        if (kTrain) {
          const int slab = (warp - kWarpEnc0) * kSlabBytes2;
          bulk_s2g(stash_tile + prog.stash_aux_pos_off + slab, sbase + S::aux_pos + slab, kSlabBytes2);
          bulk_commit();
        }
      }
      if (!args.density_only) {
        mbar_wait_relaxed(bar_dir_empty, (titer & 1) ^ 1);
        encode_row(dir, prog.n_freqs_dir, prog.freq_dir, prog.pow2_freqs != 0, args.mask_dir,
                   sbase + S::aux_dir, row);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(bar_dir_full);
          if (kTrain) {
            const int slab = (warp - kWarpEnc0) * kSlabBytes2;
            bulk_s2g(stash_tile + prog.stash_aux_dir_off + slab, sbase + S::aux_dir + slab, kSlabBytes2);
            bulk_commit();
          }
        }
      }
      __syncwarp();
    }
    if (kTrain && lane == 0) bulk_wait0();
  } else {
    // ------------------------------------------------ epilogue
    const int quarter = warp & 3, half = warp >> 2;
    const int row = quarter * 32 + lane;
    const uint32_t tmem_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const uint32_t stage_base = sbase + S::staging + quarter * (kStageBufs * kSlabBytes2);
    const bool issuer = kTrain && half == 0 && lane == 0;
    uint32_t acc_phase = 0;  // bit r: parity of accumulator region r (a register, not a local array)
    uint32_t n_staged = 0;
    uint32_t titer = 0;
    for (int64_t tile; (tile = seq.get(titer)) >= 0; ++titer) {
      const int64_t p = tile * kTileM + row;
      const bool valid = p < args.n_samples;
      uint8_t* stash_tile = kTrain ? args.stash + (size_t)tile * prog.stash_tile_bytes : nullptr;
      float sigma = 0.f;
      for (int g = 0; g < n_gemm; ++g) {
        const GemmLayer& L = prog.layer[g];
        const int r = g & 1;
        const uint32_t region = tmem_lane + (uint32_t)r * 256u;
        const bool last = (g == n_gemm - 1);
        const int epi = L.epi;
        const int nchunk = L.n_halves * 2;
        // this layer's ReLU mask words in the tile's stash record (null: the layer has none)
        uint8_t* const mask_tile = (kTrain && L.mask_off >= 0) ? stash_tile + L.mask_off : nullptr;
        if (threadIdx.x == 0) FS_TRACE2(titer, g, 3);
        mbar_wait(bar_acc_full + 8 * r, (acc_phase >> r) & 1u);
        acc_phase ^= 1u << r;
        tc_fence_after();
        if (threadIdx.x == 0) FS_TRACE2(titer, g, 4);
        float part[3] = {0.f, 0.f, 0.f};
        float sig_part = 0.f;
        // rolled on purpose: the kernel's hot loops must stay instruction-cache resident
        // (the MMA issue loop shares the SM's I-cache with this code).  Pipelining the
        // accumulator loads one chunk ahead through a second register buffer (as the dgrad
        // epilogue does) was measured SLOWER here, twice: 1.54 -> 1.71 ms per training forward in
        // round 1, 1.65 -> 1.85 ms (inference 13.1 -> 13.4 ms per 12.6 M samples) after the MMA issue fix.
#pragma unroll 1
        for (int c = 0; c < nchunk; ++c) {
          const int c0 = 64 * c + 32 * half;  // first feature handled by this thread
          uint32_t v[32];
          tmem_ld32(region + c0, v);
          float4 b4[8];
          {
            const float4* __restrict__ sb = reinterpret_cast<const float4*>(smem + S::bias) + ((g * 256 + c0) >> 2);
#pragma unroll
            for (int i = 0; i < 8; ++i) b4[i] = sb[i];
          }
          tmem_ld_wait();
          uint32_t w[16];
          if (epi == EPI_RELU || epi == EPI_CONN) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float s0, s1, s2, s3;
              add_f32x2(s0, s1, __uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), b4[i].x, b4[i].y);
              add_f32x2(s2, s3, __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]), b4[i].z, b4[i].w);
              w[2 * i] = (epi == EPI_RELU) ? pack_bf16x2_relu(s0, s1) : pack_bf16x2(s0, s1);
              w[2 * i + 1] = (epi == EPI_RELU) ? pack_bf16x2_relu(s2, s3) : pack_bf16x2(s2, s3);
            }
          } else {
            // last hidden layer (+ sigma head) / branch layer (+ rgb head): heads on CUDA cores
            const float* hw = reinterpret_cast<const float*>(smem + S::heads) + (epi == EPI_RELU_SIGMA ? 0 : 256) + c0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float h0 = fmaxf(__uint_as_float(v[4 * i]) + b4[i].x, 0.f);
              const float h1 = fmaxf(__uint_as_float(v[4 * i + 1]) + b4[i].y, 0.f);
              const float h2 = fmaxf(__uint_as_float(v[4 * i + 2]) + b4[i].z, 0.f);
              const float h3 = fmaxf(__uint_as_float(v[4 * i + 3]) + b4[i].w, 0.f);
              w[2 * i] = pack_bf16x2(h0, h1);
              w[2 * i + 1] = pack_bf16x2(h2, h3);
              const float4 w0 = *reinterpret_cast<const float4*>(hw + 4 * i);
              if (epi == EPI_RELU_SIGMA) {
                sig_part = fmaf(h0, w0.x, fmaf(h1, w0.y, fmaf(h2, w0.z, fmaf(h3, w0.w, sig_part))));
              } else {
                const float4 w1 = *reinterpret_cast<const float4*>(hw + 128 + 4 * i);
                const float4 w2 = *reinterpret_cast<const float4*>(hw + 256 + 4 * i);
                part[0] = fmaf(h0, w0.x, fmaf(h1, w0.y, fmaf(h2, w0.z, fmaf(h3, w0.w, part[0]))));
                part[1] = fmaf(h0, w1.x, fmaf(h1, w1.y, fmaf(h2, w1.z, fmaf(h3, w1.w, part[1]))));
                part[2] = fmaf(h0, w2.x, fmaf(h1, w2.y, fmaf(h2, w2.z, fmaf(h3, w2.w, part[2]))));
              }
            }
          }
          if (!last) {
            // bf16 pairs back into TMEM over the first 16 of the 32 fp32 columns just read
            tmem_st16(region + c0, w);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_a_ready + 8 * c);
          }
          if (kTrain) {
            if (mask_tile) {
              // 1-bit ReLU mask of these 32 features (what dgrad reads instead of the activations):
              // one word per row, 128 B per warp store
              uint32_t bits = 0;
#pragma unroll
              for (int q = 0; q < 16; ++q) bits = relu_bits_fold(bits, w[q], q);
              *reinterpret_cast<uint32_t*>(mask_tile + relu_bits_word_off(c, half, row)) = bits;
            }
            // SW128 image slab of this quarter's 32 rows of chunk c -> stash
            const uint32_t buf = stage_base + (n_staged % kStageBufs) * kSlabBytes2;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              st_shared_v4(buf + lane * 128 + (((uint32_t)(4 * half + j) ^ (uint32_t)(lane & 7)) << 4),
                           w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
            fence_proxy_async_smem();
            if (issuer) bulk_wait_read1();  // slabs older than the previous one have been read
            named_bar_sync(1 + quarter, 64);
            if (issuer) {
              bulk_s2g(stash_tile + L.stash_off + c * kChunkBytes + quarter * kSlabBytes2, buf, kSlabBytes2);
              bulk_commit();
            }
            ++n_staged;
          }
        }
        if (threadIdx.x == 0) FS_TRACE2(titer, g, 5);
        if (last && tab.drained_off) {  // every load of the last accumulator has completed (tmem_ld_wait)
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(sbase + tab.drained_off);
        }
        if (epi == EPI_RELU_SIGMA) {
          if (half == 1) exch[row].w = sig_part;
          named_bar_sync(1 + quarter, 64);
          if (half == 0) sigma = sig_part + exch[row].w + head_b[0];
          // density_only: 1 -> out [P]; 2 -> the sigma slot of a [P,4] (rgb, sigma) buffer
          if (last && half == 0 && valid) args.out[args.density_only == 2 ? 4 * p + 3 : p] = sigma;
        } else if (epi == EPI_BRANCH) {
          if (half == 1) {
            exch[row].x = part[0]; exch[row].y = part[1]; exch[row].z = part[2];
          }
          named_bar_sync(1 + quarter, 64);
          if (half == 0 && valid) {
            const float4 e = exch[row];
            const float z0 = part[0] + e.x + head_b[1];
            const float z1 = part[1] + e.y + head_b[2];
            const float z2 = part[2] + e.z + head_b[3];
            reinterpret_cast<float4*>(args.out)[p] =
                make_float4(1.0f / (1.0f + expf(-z0)), 1.0f / (1.0f + expf(-z1)), 1.0f / (1.0f + expf(-z2)), sigma);
          }
        }
      }
    }
    if (issuer) bulk_wait0();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kWarpMma) tmem_dealloc(tmem_base, kTmemCols2);
}

}  // namespace

int mlp_forward_v2(const MlpProgram& P, const void* packed, int64_t n_samples, int samples_per_ray,
                   const float* rays_o, const float* rays_d, const float* t_starts, const float* t_ends,
                   const float* x, const float* dirs, const float* mask_pos, const float* mask_dir,
                   int density_only, float* out, void* stash, void* stream) {
  {  // function attributes are per device
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
      cudaError_t e1 = cudaFuncSetAttribute(mlp_fwd2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            Smem<false>::total);
      cudaError_t e2 = cudaFuncSetAttribute(mlp_fwd2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            Smem<true>::total);
      for (cudaError_t e : {e1, e2})
        if (e != cudaSuccess) {
          fsnerf_set_error("mlp_forward: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
          return FSNERF_ERR_CUDA;
        }
      if (dev >= 0 && dev < 64) configured[dev] = true;
    }
  }
  Fwd2Args a;
  a.trace = reinterpret_cast<long long*>(fsnerf_debug_trace_ptr());
  a.packed = reinterpret_cast<const uint8_t*>(packed);
  a.n_samples = n_samples; a.samples_per_ray = samples_per_ray;
  a.rays_o = rays_o; a.rays_d = rays_d; a.t_starts = t_starts; a.t_ends = t_ends;
  a.x = x; a.dirs = dirs; a.mask_pos = mask_pos; a.mask_dir = mask_dir;
  a.density_only = density_only; a.out = out; a.stash = reinterpret_cast<uint8_t*>(stash);
  FS_REQUIRE(P.n_gemm <= kMaxLayers2, "mlp_forward: at most %d GEMM layers are supported", kMaxLayers2);
  const int64_t n_tiles = (n_samples + kTileM - 1) / kTileM;
  IssueTable T;
  T.drained_off = 0;
  {
    const bool train = stash != nullptr;
    const int n_gemm = density_only ? P.n_hidden : P.n_gemm;
    int last_pos_user = 0, n_cons = 0;
    for (int g = 0; g < P.n_hidden; ++g)
      if (P.layer[g].use_aux) last_pos_user = g;
    for (int g = 0; g < n_gemm; ++g)
      if (P.layer[g].n_act_chunks) ++n_cons;
    auto bar = [&](int off_train, int off_infer) { return (uint32_t)(train ? off_train : off_infer); };
    int j = 0, cons = 0;
    for (int g = 0; g < n_gemm; ++g) {
      const GemmLayer& L = P.layer[g];
      const int nch = L.n_act_chunks + L.use_aux;
      const bool is_dir = (L.epi == EPI_BRANCH);
      FS_REQUIRE(j + nch <= kMaxChunks2, "mlp_forward: more than %d K chunks per tile", kMaxChunks2);
      for (int i = 0; i < nch; ++i, ++j) {
        const int c = i - L.use_aux;  // -1: the encoding chunk (first; it is the layer's LAST block)
        IssueRec& R = T.rec[j];
        R.flags = ((uint32_t)g << 24) | ((g & 1) ? kRecDcol : 0u) | (i == 0 ? kRecFirst : 0u) |
                  (i == nch - 1 ? kRecLast : 0u);
        R.xbar = 0;
        if (c >= 0) {
          // a_ready[c] completes once per TMEM-fed layer: index = tile_iter * n_cons + cons
          R.flags |= kRecTmem | ((uint32_t)(cons & 1) << kRecParShift) | ((n_cons & 1) ? kRecParTile : 0u);
          R.a0 = (uint32_t)((g + 1) & 1) * 256u + 64u * c;
          R.abar = bar(Bars<true>::a_ready, Bars<false>::a_ready) + 8 * c;
        } else {
          R.flags |= kRecParTile;  // encoding tiles: once per tile
          R.a0 = is_dir ? bar(Smem<true>::aux_dir, Smem<false>::aux_dir) : bar(Smem<true>::aux_pos, Smem<false>::aux_pos);
          R.abar = is_dir ? bar(Bars<true>::dir_full, Bars<false>::dir_full)
                          : bar(Bars<true>::pos_full, Bars<false>::pos_full);
          if (is_dir) R.xbar = bar(Bars<true>::dir_empty, Bars<false>::dir_empty);
          else if (g == last_pos_user) R.xbar = bar(Bars<true>::pos_empty, Bars<false>::pos_empty);
        }
        R.idesc = umma_idesc_bf16(128, L.n_halves == 2 ? 256 : 128, 0, 0);
        R.accbar = bar(Bars<true>::acc_full, Bars<false>::acc_full) + 8 * (g & 1);
        R.n_acc = issue_n_acc(i, nch);
        R.w_block = (uint32_t)(L.first_block + (c >= 0 ? c : L.n_act_chunks) * L.n_halves);
        R.w_bytes = (uint32_t)L.n_halves * kBlockBytes;
        R.pad[0] = R.pad[1] = R.pad[2] = 0;
      }
      if (L.n_act_chunks) ++cons;
    }
    T.n = j;
    // A tile's first layers (layer 0, then layer 1 if its encoding chunk comes first) are issued
    // before any chunk waits for an epilogue of the tile.  The one of them that writes the
    // accumulator region of the last layer (region (n_gemm - 1) & 1: layer 0 when n_gemm is odd)
    // must wait until the epilogue has read the previous tile's last accumulator.
    for (int k = 0; k < T.n && !(T.rec[k].flags & kRecTmem); ++k)
      if ((int)((T.rec[k].flags >> 24) & 1u) == ((n_gemm - 1) & 1)) {
        T.rec[k].flags |= kRecDrained;
        T.drained_off = bar(Bars<true>::drained, Bars<false>::drained);
      }
    T.last_acc_off = bar(Bars<true>::acc_full, Bars<false>::acc_full) + 8 * ((n_gemm - 1) & 1);
    T.last_acc_n = 0;
    for (int g = 0; g < n_gemm; ++g)
      if ((g & 1) == ((n_gemm - 1) & 1)) ++T.last_acc_n;
  }
  const int grid = (int)(n_tiles < kNumSMs ? n_tiles : kNumSMs);
  FsProfScope prof_(stash ? "mlp_fwd_train" : "mlp_fwd", stream);
  if (stash)
    mlp_fwd2_kernel<true><<<grid, kThreads2, Smem<true>::total, (cudaStream_t)stream>>>(P, a, T);
  else
    mlp_fwd2_kernel<false><<<grid, kThreads2, Smem<false>::total, (cudaStream_t)stream>>>(P, a, T);
  return fsnerf_check_launch("mlp_forward");
}

}  // namespace fs

using namespace fs;

extern "C" int fsnerf_mlp_forward(const fsnerf_net_cfg* cfg, const float* params,
                                  const void* packed, int64_t n_samples, int samples_per_ray,
                                  const float* rays_o, const float* rays_d, const float* t_starts,
                                  const float* t_ends, const float* x, const float* dirs,
                                  const float* mask_pos, const float* mask_dir, int density_only,
                                  float* out, void* stash, void* stream) {
  MlpProgram P;
  int rc = build_program(cfg, &P);
  if (rc != FSNERF_OK) return rc;
  FS_REQUIRE(n_samples >= 0, "mlp_forward: negative n_samples");
  FS_REQUIRE(density_only >= 0 && density_only <= 2, "mlp_forward: density_only must be 0, 1 or 2");
  if (n_samples == 0) return FSNERF_OK;
  FS_REQUIRE(params && packed && out, "mlp_forward: null pointer");
  if (x) {
    FS_REQUIRE(density_only || dirs, "mlp_forward: dirs required unless density_only");
  } else {
    FS_REQUIRE(rays_o && rays_d && t_starts && t_ends && samples_per_ray > 0,
               "mlp_forward: rays/t_starts/t_ends required when x is NULL");
  }
  FS_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0 &&
                 (reinterpret_cast<uintptr_t>(params) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(stash) & 127) == 0,
             "mlp_forward: params/out must be 16B aligned, packed/stash 128B aligned");
  FS_REQUIRE(!(stash && density_only), "mlp_forward: stash (training) needs the full network");
  return mlp_forward_v2(P, packed, n_samples, samples_per_ray, rays_o, rays_d, t_starts, t_ends, x, dirs,
                        mask_pos, mask_dir, density_only, out, stash, stream);
}
