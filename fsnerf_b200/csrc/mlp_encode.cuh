// Frequency-masked positional encoding of one sample row into a [128 x 64] bf16
// SWIZZLE_128B operand tile (kernel (2), fused into the MLP's A-operand staging).
#pragma once
#include "common.cuh"
#include "mlp_common.cuh"

namespace fs {

// out of line on purpose: sincosf's argument reduction is ~150 instructions and the fused
// MLP kernels must keep their hot loops instruction-cache resident
static __device__ __noinline__ void sincos_acc(float x, float* sn, float* cs) { sincosf(x, sn, cs); }

// sin/cos encoding of v[3] -> 64 bf16 channels (zero padded) into row `row` of a
// [128 x 64] SW128 tile at smem address `tile`.
// reference: src/core/models.py:43-50 (channel order x, sin(f0 x), cos(f0 x), ...)
// Each channel is rounded to bf16 (round to nearest, as cvt.rn.bf16x2) as soon as it is known and
// kept as 32 packed words: 64 live fp32 channels across the out-of-line sincosf calls spilled in
// the 96-register training launch.
static __device__ __noinline__ void encode_row(const float v[3], int n_freqs, const float* freqs, bool pow2,
                                           const float* __restrict__ mask, uint32_t tile, int row) {
  uint32_t pk[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) pk[i] = 0u;
  // channel i (i < 3 + 6 n_freqs: the mask, if any, applies)
  auto put = [&](int i, float x) {
    if (mask) x *= __ldg(mask + i);
    pk[i >> 1] |= (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(x)) << (16 * (i & 1));
  };
  put(0, v[0]); put(1, v[1]); put(2, v[2]);
  if (pow2) {
    // f_k = 2^k (log_space, the reference default): an accurate sincosf every 4th octave,
    // exact double-angle steps (sin 2a = 2 s c, cos 2a = 1 - 2 s^2) in between.  The error
    // doubles per step, so it stays <= ~8 ulp (1e-6) — invisible after the bf16 rounding.
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      float sn = 0.f, cs = 1.f;
#pragma unroll
      for (int k = 0; k < kMaxFreqs; ++k) {
        if (k < n_freqs) {
          if ((k & 3) == 0) {
            sincos_acc(v[a] * freqs[k], &sn, &cs);
          } else {
            const float s2 = 2.0f * sn * cs;
            cs = fmaf(-2.0f * sn, sn, 1.0f);
            sn = s2;
          }
          put(3 + 6 * k + a, sn);
          put(3 + 6 * k + 3 + a, cs);
        }
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < kMaxFreqs; ++k) {
      if (k < n_freqs) {
        float f = freqs[k];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          float sn, cs;
          sincos_acc(v[a] * f, &sn, &cs);
          put(3 + 6 * k + a, sn);
          put(3 + 6 * k + 3 + a, cs);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st_shared_v4(tile + sw128_off(row, j), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
}

}  // namespace fs
