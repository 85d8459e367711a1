// Shared machinery of the tensor-memory-resident MLP kernels (mlp_fwd2.cu, mlp_bwd2.cu):
// the per-tile chunk table, the two alternating MMA-issuer warps and the weight producers.
//
// What the hardware dictated (tools/mma_bench.cu, tools/l2_bench.cu, measured on B200):
//  * a tcgen05.mma blocks at issue until the previous MMA has (nearly) finished and the
//    tensor pipe idles whenever no MMA is waiting at that point; M=128 N=256 K=16 runs at
//    128 cycles when the issue stream is dense enough.  One warp cannot do a chunk's
//    bookkeeping (operand waits, descriptors, commits: 400+ cycles of dependent
//    uniform-datapath instructions) inside the 512 cycles of its four MMAs, so TWO warps
//    alternate chunks and pass a token right after their last MMA issue.
//  * tcgen05 instructions take their operands from UNIFORM registers.  Issued under a per-lane
//    guard (`@lane0 tcgen05.mma`, or inside `if (lane == 0)`) the compiler cannot know that one
//    thread is active and wraps EVERY instruction in an ELECT + 6x R2UR.BROADCAST loop: ~160
//    cycles per MMA at issue, above the 128 it takes to execute (round 1 and most of round 2
//    shipped that: 650 cycles per 64-wide K chunk instead of 512).  Inside `if (elect_one())`
//    (elect.sync) the operands move with plain R2UR ahead of four back-to-back UTCHMMA: the
//    inference forward went from 14.0 to 12.7 ms per 12.6 M samples (76 % -> 84 % of the sustained
//    bf16 peak).  The chunk table is a __grid_constant__ kernel parameter (uniform loads), the
//    waits exit on warp votes, the warp index comes from a shuffle.
//  * bulk copies issued by one thread do not overlap (~440 cycles each, any size <= 32 KB):
//    two producer warps, 32 KB stages.
#pragma once
#include "common.cuh"
#include "mlp_common.cuh"

namespace fs {

constexpr int kMaxChunks2 = 64;          // K chunks per tile in the issue table
constexpr int kMmaWarps = 2;             // MMA issuers, alternating K chunks
constexpr int kProdWarps = 2;            // weight producers, alternating stages
constexpr int kStageBytes = 2 * kBlockBytes;  // one [256 x 64] bf16 operand stage

// record flags
constexpr uint32_t kRecDcol = 0x100u;        // accumulator region: TMEM column offset 0 / 256
constexpr uint32_t kRecTmem = 1u << 16;      // A operand from tensor memory (else an smem SW128 tile)
constexpr uint32_t kRecFirst = 1u << 17;     // first chunk of its layer: overwrite the accumulator
constexpr uint32_t kRecParTile = 1u << 18;   // operand-barrier parity toggles with the tile iteration
constexpr uint32_t kRecParShift = 19;        // bit 19: base parity of the operand barrier
constexpr uint32_t kRecLast = 1u << 20;      // last chunk of its layer (trace only)
// the chunk overwrites the accumulator region of the previous tile's last layer before any chunk
// of its tile has waited for an epilogue: wait until the epilogue has read that accumulator
constexpr uint32_t kRecDrained = 1u << 21;

// One record per 64-wide K chunk of a tile, in consumption order.  The table is a kernel
// parameter so the issuing warps read it with uniform loads.
struct IssueRec {
  uint32_t flags;    // kRec* | layer << 24
  uint32_t idesc;
  uint32_t a0;       // TMEM column of the chunk's A operand, or smem byte offset of the A tile
  uint32_t abar;     // smem byte offset of the operand-ready barrier
  uint32_t xbar;     // smem byte offset of an "A tile free" barrier to commit after the chunk (0: none)
  uint32_t accbar;   // smem byte offset of the accumulator-full barrier
  uint32_t n_acc;    // how many times to commit it after this chunk (it expects one commit per issuer)
  uint32_t w_block;  // first 16 KB block of the chunk's B operand in the packed image
  uint32_t w_bytes;  // bytes of that operand (32 KB for N = 256, 16 KB for N = 128)
  uint32_t pad[3];
};
struct IssueTable {
  int n;
  uint32_t last_acc_off;  // accumulator-full barrier of the tile's last layer (smem byte offset)
  uint32_t last_acc_n;    // layers per tile sharing that barrier
  // barrier the epilogue completes once per tile after reading the last layer's accumulator, which
  // kRecDrained chunks wait for (smem byte offset; 0: no chunk needs it)
  uint32_t drained_off;
  IssueRec rec[kMaxChunks2];
};

// Host side: accumulator-full commits.  Chunks alternate between the two issuers, so the
// last chunk's issuer commits once and the previous chunk's issuer once; the issuer of a
// single-chunk layer commits twice.
inline uint32_t issue_n_acc(int i, int nch) {
  return (i == nch - 1) ? (nch == 1 ? 2u : 1u) : (i == nch - 2 ? 1u : 0u);
}

struct IssueBars {
  uint32_t w_full, w_empty, token;  // smem addresses: [kStages], [kStages], [2]
  uint32_t ring;                    // smem address of the operand ring
};

// ------------------------------------------------------------------ 1-bit ReLU masks
// One 32-bit word per (sample row, 32-column half of a 64-feature chunk).  Pair q of the half
// (columns 2q, 2q+1, the bf16x2 word w[q] of the epilogues) owns bits 15-q and 31-q, so that
// `word << q` puts them on the sign bits of bytes 1 and 3, where ONE PRMT with sign replication
// expands them into the 0xFFFF / 0x0000 AND-mask of a packed bf16x2 gradient.
// forward: fold pair q's non-zero flags into the word (h = two post-ReLU bf16, sign bits clear:
// h + 0x7FFF per half sets that half's top bit iff it is non-zero; no carry since h <= 0x7FFF)
__device__ __forceinline__ uint32_t relu_bits_fold(uint32_t word, uint32_t h, int q) {
  return word | (((h + 0x7FFF7FFFu) & 0x80008000u) >> q);
}
// backward: AND-mask of pair q
__device__ __forceinline__ uint32_t relu_bits_mask2(uint32_t word, int q) {
  uint32_t r;
  asm("prmt.b32 %0, %1, 0, 0xBB99;" : "=r"(r) : "r"(word << q));
  return r;
}
__host__ __device__ __forceinline__ uint32_t relu_bits_word_off(int chunk, int half, int row) {
  return (uint32_t)(((chunk * 2 + half) * kTileM + row) * 4);
}

// ------------------------------------------------------------------ tile sequence of a CTA
// Static: n_iters tiles first, first + stride, ...  Dynamic (feed != nullptr): one thread of the
// CTA claims tiles from a global counter a little ahead of their use and publishes them in shared
// memory: feed[0] = tiles claimed so far (monotonic), feed[1 + (i & 3)] = tile of iteration i or -1
// when the work has run out.  Every role warp asks for iteration i and gets the same answer.
struct TileSeq {
  volatile int* feed;
  int64_t first, stride, n_tiles;
  int64_t n_iters;  // static sequences only
  __device__ __forceinline__ static TileSeq strided(int64_t first, int64_t stride, int64_t n_tiles) {
    const int64_t n = first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0;
    return TileSeq{nullptr, first, stride, n_tiles, n};
  }
  __device__ __forceinline__ int64_t get(uint32_t titer) const {
    if (feed == nullptr) return (int64_t)titer < n_iters ? first + (int64_t)titer * stride : -1;
    uint32_t spins = 0;
    while (feed[0] <= (int)titer) {
      __nanosleep(32);
      if (++spins > (1u << 24)) { printf("fsnerf: tile feed timeout blk %d thr %d\n", blockIdx.x, threadIdx.x); __trap(); }
    }
    return feed[1 + (titer & 3u)];
  }
  // "is there a tile for iteration titer", for a warp that must stay provably converged (the MMA
  // issuers): exits and result are warp votes
  __device__ __forceinline__ bool has_converged(uint32_t titer) const {
    if (feed == nullptr) return (int64_t)titer < n_iters;
    uint32_t spins = 0;
    while (!__all_sync(0xffffffffu, feed[0] > (int)titer)) {
      if (++spins > (1u << 26)) {
        if ((threadIdx.x & 31) == 0) printf("fsnerf: tile feed timeout blk %d thr %d\n", blockIdx.x, threadIdx.x);
        __trap();
      }
    }
    return __all_sync(0xffffffffu, feed[1 + (titer & 3u)] >= 0);
  }
};

// ------------------------------------------------------------------ weight producers
// Producer `me` of kProdWarps streams every kProdWarps-th stage: L2 -> smem, one bulk copy.
template <int kStages>
__device__ __forceinline__ void producer_loop(const IssueTable& tab, const IssueBars& B, const uint8_t* packed,
                                              const TileSeq& seq, int me, int lane) {
  uint32_t cnt = 0;
  for (uint32_t titer = 0; seq.get(titer) >= 0; ++titer) {
    for (int j = 0; j < tab.n; ++j, ++cnt) {
      if ((int)(cnt % kProdWarps) != me) continue;
      const uint32_t stage = cnt % kStages, phase = (cnt / kStages) & 1;
      mbar_wait_relaxed(B.w_empty + 8 * stage, phase ^ 1);
      if (lane == 0) {
        const uint32_t bytes = tab.rec[j].w_bytes;
        mbar_arrive_expect_tx(B.w_full + 8 * stage, bytes);
        bulk_g2s(B.ring + stage * kStageBytes, packed + (size_t)tab.rec[j].w_block * kBlockBytes, bytes,
                 B.w_full + 8 * stage);
      }
      __syncwarp();
    }
  }
}

// Single-thread form: thread `me` of kProdWarps issuing threads (lanes of ONE warp, each on its
// own divergent path) streams every kProdWarps-th stage.
template <int kStages>
__device__ __forceinline__ void producer_loop_thread(const IssueTable& tab, const IssueBars& B, const uint8_t* packed,
                                                     const TileSeq& seq, int me) {
  uint32_t cnt = 0;
  for (uint32_t titer = 0; seq.get(titer) >= 0; ++titer) {
    for (int j = 0; j < tab.n; ++j, ++cnt) {
      if ((int)(cnt % kProdWarps) != me) continue;
      const uint32_t stage = cnt % kStages, phase = (cnt / kStages) & 1;
      mbar_wait_relaxed(B.w_empty + 8 * stage, phase ^ 1);
      const uint32_t bytes = tab.rec[j].w_bytes;
      mbar_arrive_expect_tx(B.w_full + 8 * stage, bytes);
      bulk_g2s(B.ring + stage * kStageBytes, packed + (size_t)tab.rec[j].w_block * kBlockBytes, bytes,
               B.w_full + 8 * stage);
    }
  }
}

// ------------------------------------------------------------------ MMA issuers
// All 32 lanes of issuer `me` run this loop in lock step on provably uniform values; the
// tcgen05 instructions are guarded so that lane 0 alone issues them.  trace: optional
// clock64 timeline [tile iteration < 4][layer][k]: k = 0 layer reached, 1 first MMA, 2 committed.
template <int kStages>
__device__ __forceinline__ void issuer_loop(const IssueTable& tab, const IssueBars& B, uint32_t sbase,
                                            const TileSeq& seq, uint32_t me, int lane, long long* trace) {
  const int n_rec = tab.n;
  uint32_t titer = 0;
  int j = (int)me;
  if (j >= n_rec) { j -= n_rec; ++titer; }
  bool more = seq.has_converged(titer);
  uint32_t stage = me % kStages, wpar = 0, tok_par = me ? 0u : 1u;
  const bool tr = trace != nullptr && blockIdx.x == 0 && lane == 0;
  while (more) {
    const IssueRec& R = tab.rec[j];
    const uint32_t flags = R.flags, idesc = R.idesc;
    const bool is_tmem = flags & kRecTmem, first = flags & kRecFirst;
    const uint32_t d_col = flags & kRecDcol;
    const uint32_t g_cur = flags >> 24;
    const uint32_t a0 = is_tmem ? R.a0 : umma_desc_lo(sbase + R.a0);
    const uint32_t b0 = umma_desc_lo(B.ring + stage * kStageBytes);
    const uint32_t apar = (((flags & kRecParTile) ? titer : 0u) ^ (flags >> kRecParShift)) & 1u;
    if (tr && first && titer < 4) trace[(titer * 16 + g_cur) * 8 + 0] = clock64();
    mbar_wait_converged(B.w_full + 8 * stage, wpar);
    mbar_wait_converged(sbase + R.abar, apar);
    if ((flags & kRecDrained) && titer > 0) mbar_wait_converged(sbase + tab.drained_off, (titer - 1) & 1u);
    mbar_wait_converged(B.token + 8 * me, tok_par);  // the other issuer has queued its chunk
    tok_par ^= 1u;
    tc_fence_after();
    if (tr && first && titer < 4) trace[(titer * 16 + g_cur) * 8 + 1] = clock64();
    const uint32_t n_acc = R.n_acc;
    const uint32_t acc0 = first ? 0u : 1u;
    if (elect_one()) {  // one thread issues the chunk's MMAs, the hand-over and the completion arrivals
      if (is_tmem) {  // features [0,32) of the chunk at columns +0, +8; [32,64) at +32, +40
        umma_bf16_ts(d_col, a0, umma_desc_from_lo(b0), idesc, acc0);
        umma_bf16_ts(d_col, a0 + 8, umma_desc_from_lo(b0 + 2), idesc, 1u);
        umma_bf16_ts(d_col, a0 + 32, umma_desc_from_lo(b0 + 4), idesc, 1u);
        umma_bf16_ts(d_col, a0 + 40, umma_desc_from_lo(b0 + 6), idesc, 1u);
      } else {
        umma_bf16_ss(d_col, umma_desc_from_lo(a0), umma_desc_from_lo(b0), idesc, acc0);
        umma_bf16_ss(d_col, umma_desc_from_lo(a0 + 2), umma_desc_from_lo(b0 + 2), idesc, 1u);
        umma_bf16_ss(d_col, umma_desc_from_lo(a0 + 4), umma_desc_from_lo(b0 + 4), idesc, 1u);
        umma_bf16_ss(d_col, umma_desc_from_lo(a0 + 6), umma_desc_from_lo(b0 + 6), idesc, 1u);
      }
      mbar_arrive(B.token + 8 * (me ^ 1u));  // the last MMA is queued: hand over
      umma_commit(B.w_empty + 8 * stage);
      if (R.xbar) umma_commit(sbase + R.xbar);
      if (n_acc) {
        umma_commit(sbase + R.accbar);
        if (n_acc > 1) umma_commit(sbase + R.accbar);
      }
    }
    __syncwarp();
    if (n_acc && tr && (flags & kRecLast) && titer < 4) trace[(titer * 16 + g_cur) * 8 + 2] = clock64();
    // next chunk of mine
    j += kMmaWarps;
    stage += kMmaWarps;
    if (stage >= (uint32_t)kStages) { stage -= kStages; wpar ^= 1u; }
    if (j >= n_rec) {
      j -= n_rec;
      more = seq.has_converged(titer + 1);
      // the next tile's first layer overwrites TMEM region 0, which the last layer still reads
      // as its A operand: let the tensor pipe drain first (that barrier completes last_acc_n
      // times per tile)
      if (more) mbar_wait_converged(sbase + tab.last_acc_off, ((titer + 1) * tab.last_acc_n - 1) & 1u);
      ++titer;
    }
  }
}

}  // namespace fs
