// Host side of the fused MLP: program construction, operand packing.
#include <math.h>
#include <string.h>
#include "common.cuh"
#include "mlp_common.cuh"

namespace fs {

int build_program(const fsnerf_net_cfg* cfg, MlpProgram* P) {
  FS_REQUIRE(cfg && P, "net cfg: null");
  FS_REQUIRE(cfg->d_hidden == 256, "net cfg: d_hidden must be 256 (tcgen05 tile width), got %d",
             cfg->d_hidden);
  FS_REQUIRE(cfg->n_layers >= 2 && cfg->n_layers <= kMaxHidden, "net cfg: n_layers must be in [2,%d], got %d",
             kMaxHidden, cfg->n_layers);
  FS_REQUIRE(cfg->n_freqs_pos >= 0 && cfg->n_freqs_pos <= kMaxFreqs, "net cfg: n_freqs_pos must be <= 10");
  FS_REQUIRE(cfg->n_freqs_dir >= 0 && cfg->n_freqs_dir <= kMaxFreqs, "net cfg: n_freqs_dir must be <= 10");
  FS_REQUIRE((cfg->skip_mask >> (cfg->n_layers - 1)) == 0,
             "net cfg: skip on or after the last hidden layer is unsupported");
  memset(P, 0, sizeof(*P));
  const int H = cfg->d_hidden, n = cfg->n_layers;
  P->n_hidden = n;
  P->n_freqs_pos = cfg->n_freqs_pos;
  P->n_freqs_dir = cfg->n_freqs_dir;
  P->pow2_freqs = cfg->log_space ? 1 : 0;
  P->d_pos = 3 * (1 + 2 * cfg->n_freqs_pos);
  P->d_dir = 3 * (1 + 2 * cfg->n_freqs_dir);
  // frequencies exactly as torch builds them (src/core/models.py:30-34)
  for (int pass = 0; pass < 2; ++pass) {
    int L = pass ? cfg->n_freqs_dir : cfg->n_freqs_pos;
    float* f = pass ? P->freq_dir : P->freq_pos;
    for (int k = 0; k < L; ++k) {
      if (cfg->log_space) {
        f[k] = ldexpf(1.0f, k);
      } else {
        // torch.linspace(1, 2^(L-1), L): symmetric evaluation around the midpoint
        float start = 1.0f, end = ldexpf(1.0f, L - 1);
        float step = (L > 1) ? (end - start) / (float)(L - 1) : 0.0f;
        f[k] = (k < L / 2) ? start + step * (float)k : end - step * (float)(L - 1 - k);
      }
    }
  }
  int64_t off = 0;
  auto al4 = [](int64_t v) { return (v + 3) & ~(int64_t)3; };
  int n_t = 0;
  auto tensor = [&](int64_t numel) {  // next tensor in state-dict order, 16 B aligned
    off = al4(off);
    int64_t o = off;
    P->tensor_off[n_t] = o;
    P->tensor_numel[n_t] = numel;
    ++n_t;
    off += numel;
    return (int)o;
  };
  int blk = 0;
  int stash = 0;
  P->stash_aux_pos_off = stash;
  stash += kChunkBytes;
  int g = 0;
  for (int i = 0; i < n; ++i, ++g) {
    GemmLayer& L = P->layer[g];
    bool first = (i == 0);
    bool skip_in = !first && ((cfg->skip_mask >> (i - 1)) & 1);
    L.n_act_chunks = first ? 0 : H / 64;
    L.use_aux = (first || skip_in) ? 1 : 0;
    L.n_halves = H / 128;
    L.epi = (i == n - 1) ? EPI_RELU_SIGMA : EPI_RELU;
    L.ld = first ? P->d_pos : (skip_in ? H + P->d_pos : H);
    L.w_off = tensor((int64_t)H * L.ld);
    L.bias_off = tensor(H);
    L.first_block = blk;
    blk += (L.n_act_chunks + L.use_aux) * L.n_halves;
    L.stash_off = stash;
    stash += (H / 64) * kChunkBytes;
  }
  P->sigma_w_off = tensor(H);
  P->sigma_b_off = tensor(1);
  P->n_blocks_fwd_density = blk;
  {  // connection
    GemmLayer& L = P->layer[g++];
    L.n_act_chunks = H / 64; L.use_aux = 0; L.n_halves = H / 128; L.epi = EPI_CONN;
    L.ld = H; L.w_off = tensor((int64_t)H * H); L.bias_off = tensor(H);
    L.first_block = blk; blk += L.n_act_chunks * L.n_halves;
    L.stash_off = stash; stash += (H / 64) * kChunkBytes;
  }
  P->stash_aux_dir_off = stash;
  stash += kChunkBytes;
  {  // branch
    GemmLayer& L = P->layer[g++];
    L.n_act_chunks = H / 64; L.use_aux = 1; L.n_halves = (H / 2) / 128; L.epi = EPI_BRANCH;
    L.ld = H + P->d_dir; L.w_off = tensor((int64_t)(H / 2) * L.ld);
    L.bias_off = tensor(H / 2);
    L.first_block = blk; blk += (L.n_act_chunks + 1) * L.n_halves;
    L.stash_off = stash; stash += ((H / 2) / 64) * kChunkBytes;
  }
  P->rgb_w_off = tensor(3 * (H / 2));
  P->rgb_b_off = tensor(3);
  off = al4(off);
  P->n_tensors = n_t;
  P->n_gemm = g;
  P->n_blocks_fwd = blk;
  P->n_params = off;
  // 1-bit ReLU masks behind the operand images (existing offsets stay put): per layer
  // [n_out/64 chunks][2 column halves][128 rows] x 4 B
  for (int gi = 0; gi < g; ++gi) {
    GemmLayer& L = P->layer[gi];
    if (L.epi == EPI_CONN) { L.mask_off = -1; continue; }
    L.mask_off = stash;
    stash += (L.n_halves * 2) * 2 * kTileM * 4;
  }
  P->stash_tile_bytes = stash;
  // dgrad (W^T) blocks, in backward consumption order: branch, conn, hidden n-1 .. 1
  for (int gi = P->n_gemm - 1; gi >= 1; --gi) {
    GemmLayer& L = P->layer[gi];
    int n_out = L.n_halves * 128;
    L.bwd_first_block = blk;
    L.bwd_n_halves = H / 128;  // gradient w.r.t. the first d_hidden inputs only
    L.bwd_n_chunks = n_out / 64;
    blk += L.bwd_n_halves * L.bwd_n_chunks;
  }
  P->layer[0].bwd_first_block = -1;
  int dst = 0;
  for (int gi = 0; gi < P->n_gemm; ++gi) {
    P->layer[gi].dstash_off = dst;
    dst += (P->layer[gi].n_halves * 128 / 64) * kChunkBytes;
  }
  P->dstash_tile_bytes = dst;
  P->n_blocks_bwd = blk - P->n_blocks_fwd;
  FS_REQUIRE(blk <= 192, "net cfg: %d operand blocks exceed the pack table (192): fewer layers", blk);
  P->small_off = (int64_t)blk * kBlockBytes;
  P->packed_bytes = P->small_off + (int64_t)kSmallFloats * 4;
  return FSNERF_OK;
}

namespace {

struct PackBlk {
  int w_off;
  short ld, row0, col0, nrows, ncols, transposed;
};
constexpr int kMaxPackBlk = 192;
struct PackTable {
  int n;
  int n_gemm;
  int bias_off[kMaxGemm], bias_n[kMaxGemm];
  int sigma_w_off, sigma_b_off, rgb_w_off, rgb_b_off;
  PackBlk b[kMaxPackBlk];
};

__global__ void __launch_bounds__(256)
pack_kernel(const __grid_constant__ PackTable T, const float* __restrict__ params,
            uint8_t* __restrict__ packed) {
  if ((int)blockIdx.x == T.n) {  // last CTA: the contiguous fp32 small-params block
    float* sm = reinterpret_cast<float*>(packed + (size_t)T.n * kBlockBytes);
    for (int i = threadIdx.x; i < kSmallFloats; i += blockDim.x) {
      float v = 0.f;
      if (i < kSmallSigmaW) {
        int g = i >> 8, c = i & 255;
        if (g < T.n_gemm && c < T.bias_n[g]) v = params[T.bias_off[g] + c];
      } else if (i < kSmallRgbW) {
        v = params[T.sigma_w_off + (i - kSmallSigmaW)];
      } else if (i < kSmallSigmaB) {
        v = params[T.rgb_w_off + (i - kSmallRgbW)];
      } else if (i == kSmallSigmaB) {
        v = params[T.sigma_b_off];
      } else if (i < kSmallRgbB + 3) {
        v = params[T.rgb_b_off + (i - kSmallRgbB)];
      }
      sm[i] = v;
    }
    return;
  }
  const PackBlk b = T.b[blockIdx.x];
  uint8_t* dst = packed + (size_t)blockIdx.x * kBlockBytes;
  const float* W = params + b.w_off;
  for (int u = threadIdx.x; u < 1024; u += blockDim.x) {
    int i = u >> 3, j = u & 7;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      int kk = j * 8 + e;
      float x = 0.f;
      if (i < b.nrows && kk < b.ncols) {
        x = b.transposed ? W[(size_t)(b.row0 + kk) * b.ld + (b.col0 + i)]
                         : W[(size_t)(b.row0 + i) * b.ld + (b.col0 + kk)];
      }
      v[e] = x;
    }
    uint4 w4 = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                          pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    *reinterpret_cast<uint4*>(dst + sw128_off(i, j)) = w4;
  }
}

}  // namespace
}  // namespace fs

using namespace fs;

extern "C" int64_t fsnerf_mlp_param_count(const fsnerf_net_cfg* cfg) {
  MlpProgram P;
  if (build_program(cfg, &P) != FSNERF_OK) return -1;
  return P.n_params;
}
extern "C" int fsnerf_mlp_param_layout(const fsnerf_net_cfg* cfg, int64_t* offsets, int64_t* numels,
                                       int max_tensors) {
  MlpProgram P;
  int rc = build_program(cfg, &P);
  if (rc != FSNERF_OK) return rc;
  FS_REQUIRE(offsets && numels && max_tensors >= P.n_tensors, "mlp_param_layout: need room for %d tensors",
             P.n_tensors);
  for (int i = 0; i < P.n_tensors; ++i) {
    offsets[i] = P.tensor_off[i];
    numels[i] = P.tensor_numel[i];
  }
  return P.n_tensors;
}
extern "C" int64_t fsnerf_mlp_packed_bytes(const fsnerf_net_cfg* cfg) {
  MlpProgram P;
  if (build_program(cfg, &P) != FSNERF_OK) return -1;
  return P.packed_bytes;
}
extern "C" int64_t fsnerf_mlp_stash_bytes(const fsnerf_net_cfg* cfg, int64_t n_samples) {
  MlpProgram P;
  if (build_program(cfg, &P) != FSNERF_OK) return -1;
  int64_t tiles = (n_samples + kTileM - 1) / kTileM;
  return tiles * (int64_t)P.stash_tile_bytes;
}

extern "C" int fsnerf_mlp_pack(const fsnerf_net_cfg* cfg, const float* params, void* packed,
                               void* stream) {
  MlpProgram P;
  int rc = build_program(cfg, &P);
  if (rc != FSNERF_OK) return rc;
  FS_REQUIRE(params && packed, "mlp_pack: null pointer");
  FS_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0, "mlp_pack: packed must be 128B aligned");
  FS_REQUIRE(P.n_blocks_fwd + P.n_blocks_bwd <= kMaxPackBlk,
             "mlp_pack: %d operand blocks exceed the pack table (%d): fewer layers", P.n_blocks_fwd + P.n_blocks_bwd,
             kMaxPackBlk);
  PackTable T;
  T.n = 0;
  for (int g = 0; g < P.n_gemm; ++g) {
    const GemmLayer& L = P.layer[g];
    int n_out = L.n_halves * 128;
    int nchunks = L.n_act_chunks + L.use_aux;
    int n_act_cols = L.n_act_chunks * 64;
    for (int c = 0; c < nchunks; ++c)
      for (int nh = 0; nh < L.n_halves; ++nh) {
        PackBlk& b = T.b[T.n++];
        b.w_off = L.w_off; b.ld = (short)L.ld; b.transposed = 0;
        b.row0 = (short)(nh * 128); b.nrows = (short)((n_out - nh * 128) < 128 ? (n_out - nh * 128) : 128);
        b.col0 = (short)(c * 64);
        b.ncols = (short)((c < L.n_act_chunks) ? 64 : (L.ld - n_act_cols));
      }
  }
  FS_REQUIRE(T.n == P.n_blocks_fwd, "mlp_pack: internal block count mismatch (%d vs %d)", T.n, P.n_blocks_fwd);
  for (int g = P.n_gemm - 1; g >= 1; --g) {
    const GemmLayer& L = P.layer[g];
    for (int c = 0; c < L.bwd_n_chunks; ++c)
      for (int nh = 0; nh < L.bwd_n_halves; ++nh) {
        PackBlk& b = T.b[T.n++];
        b.w_off = L.w_off; b.ld = (short)L.ld; b.transposed = 1;
        b.row0 = (short)(c * 64); b.ncols = 64;   // K = output features
        b.col0 = (short)(nh * 128); b.nrows = 128;  // rows = input features
      }
  }
  FS_REQUIRE(T.n == P.n_blocks_fwd + P.n_blocks_bwd && T.n <= kMaxPackBlk,
             "mlp_pack: internal block count mismatch");
  FsProfScope prof_("mlp_pack", stream);
  T.n_gemm = P.n_gemm;
  for (int g = 0; g < P.n_gemm; ++g) {
    T.bias_off[g] = P.layer[g].bias_off;
    T.bias_n[g] = P.layer[g].n_halves * 128;
  }
  T.sigma_w_off = P.sigma_w_off; T.sigma_b_off = P.sigma_b_off;
  T.rgb_w_off = P.rgb_w_off; T.rgb_b_off = P.rgb_b_off;
  pack_kernel<<<T.n + 1, 256, 0, (cudaStream_t)stream>>>(T, params, reinterpret_cast<uint8_t*>(packed));
  return fsnerf_check_launch("mlp_pack");
}
