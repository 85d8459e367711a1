// Host/device shared description of the fused NeRF MLP "program".
//
// Data layout in HBM (DESIGN.md §3):
//  * params   fp32, flat, reference state-dict order (src/core/models.py:96-108),
//             each tensor starting on a 16 B boundary (fsnerf_mlp_param_layout).
//  * packed   bf16 operand image: a sequence of 16 KB blocks, each a
//             [128 rows x 64 K] K-major SWIZZLE_128B tile ready to be the B
//             operand of tcgen05.mma after ONE bulk copy.  Forward blocks are
//             W[n][k] (rows = output features), backward (dgrad) blocks are
//             W^T (rows = input features, K = output features).
//  * stash    per 128-sample tile, the bf16 SWIZZLE_128B images of every GEMM
//             input (exact byte image of the A operand in shared memory), so
//             that the backward kernels can bulk-load them straight back, followed
//             by the 1-bit ReLU masks of every layer output (4 KB per 256-wide layer).
#pragma once
#include <stdint.h>
#include "../../include/fsnerf_b200.h"

namespace fs {

constexpr int kTileM = 128;          // samples per tile (UMMA M)
constexpr int kBlockBytes = 16384;   // one [128 x 64] bf16 SW128 block
constexpr int kChunkBytes = 16384;   // one K-chunk of an activation tile (128 rows x 128 B)
constexpr int kMaxGemm = 16;
// hidden layers build_program accepts; n_gemm = n_layers + 2 (connection, branch) must fit the
// forward's and the backward's bias tables (static_asserts next to them)
constexpr int kMaxHidden = 10;
constexpr int kMaxFreqs = 10;        // 3*(1+2L) <= 64
// "small params" block appended to the packed image: fp32 copies of every bias and
// of the sigma / rgb head weights, contiguous so ONE device-to-device copy moves
// them into __constant__ memory (uniform operands of the epilogue FADD/FFMA).
constexpr int kSmallBias = 0;                       // [kMaxGemm][256]
constexpr int kSmallSigmaW = kMaxGemm * 256;        // [256]
constexpr int kSmallRgbW = kSmallSigmaW + 256;      // [3][128]
constexpr int kSmallSigmaB = kSmallRgbW + 384;      // [1]
constexpr int kSmallRgbB = kSmallSigmaB + 1;        // [3]
constexpr int kSmallFloats = 4864;                  // padded

enum Epi : int {
  EPI_RELU = 0,        // h = relu(acc + b) -> act
  EPI_RELU_SIGMA = 1,  // last hidden layer: as EPI_RELU, plus sigma head on CUDA cores
  EPI_CONN = 2,        // h = acc + b -> act ; view-dir encoding -> aux
  EPI_BRANCH = 3,      // h = relu(acc + b) (128 wide) ; rgb head + sigmoid on CUDA cores
};

struct GemmLayer {
  int n_act_chunks;  // K chunks taken from the act buffer (0 or d_hidden/64)
  int use_aux;       // 1: one more K chunk from the aux (encoding) buffer
  int n_halves;      // N / 128
  int epi;
  int first_block;   // first forward block of this layer in the packed image
  int bias_off;      // float offset of the bias in params
  int w_off;         // float offset of the weight in params
  int ld;            // weight row length (in_features)
  int stash_off;     // byte offset of this layer's OUTPUT image in a tile's stash record (-1: none)
  int bwd_first_block;  // first dgrad block (W^T) of this layer, -1 if no dgrad needed
  int bwd_n_halves;     // dgrad output width / 128 (2)
  int bwd_n_chunks;     // dgrad K chunks = N_out / 64
  int dstash_off;       // byte offset of d(pre-activation) image in a tile's backward record
  // byte offset, in a tile's stash record, of the 1-bit ReLU mask of this layer's OUTPUT
  // ([chunk][column half][128 rows] 32-bit words, see relu_bits_* in mlp_issue.cuh); -1: the
  // layer has no ReLU.  dgrad reads these 32 B/sample/layer instead of the 512 B activations.
  int mask_off;
};

struct MlpProgram {
  int n_gemm;          // GEMM layers executed (hidden [+ conn + branch])
  int n_hidden;
  int n_blocks_fwd;    // forward blocks streamed per tile (full program)
  int n_blocks_fwd_density;  // ... when only the hidden layers run (density_only)
  int n_blocks_bwd;
  int d_pos, d_dir;    // encoding widths (63, 27)
  int n_freqs_pos, n_freqs_dir;
  int pow2_freqs;      // 1: f_k = 2^k exactly (log_space) -> double-angle recurrence in the encoder
  float freq_pos[kMaxFreqs], freq_dir[kMaxFreqs];
  int sigma_w_off, sigma_b_off, rgb_w_off, rgb_b_off;
  int stash_aux_pos_off, stash_aux_dir_off;  // byte offsets in the tile record
  int stash_tile_bytes;
  int dstash_tile_bytes;  // backward workspace record per tile (dpre images of every GEMM layer)
  int64_t n_params;      // flat fp32 length incl. alignment padding
  int n_tensors;         // state-dict tensors (2 per Linear)
  int64_t tensor_off[2 * kMaxGemm + 8];
  int64_t tensor_numel[2 * kMaxGemm + 8];
  int64_t packed_bytes;  // operand blocks + the small-params block
  int64_t small_off;     // byte offset of the small-params block in the packed image
  GemmLayer layer[kMaxGemm];
};

// Build the program from the architecture; returns 0 or FSNERF_ERR_*.
int build_program(const fsnerf_net_cfg* cfg, MlpProgram* prog);

// second-generation forward (mlp_fwd2.cu): activations resident in tensor memory
int mlp_forward_v2(const MlpProgram& P, const void* packed, int64_t n_samples, int samples_per_ray,
                   const float* rays_o, const float* rays_d, const float* t_starts, const float* t_ends,
                   const float* x, const float* dirs, const float* mask_pos, const float* mask_dir,
                   int density_only, float* out, void* stash, void* stream);

}  // namespace fs
