// Kernel (3) backward: the NeRF MLP gradient (the loss.backward() edge of
// src/run-nerf.py:282 through src/core/models.py:111-143) as ONE persistent launch whose
// CTAs take one of two roles, plus a small SIMT kernel for the degenerate heads.
//
//  dgrad CTAs (blockIdx < n_d), tile-stationary: the fused d(pre-activation) chain of one
//    128-sample tile at a time with the gradients resident in TENSOR MEMORY (same skeleton as
//    mlp_fwd2.cu):
//      warps 0..7   epilogue: TMEM -> regs (loads pipelined one chunk ahead) -> (+ sigma-head
//                   term) -> 1-bit ReLU mask written by the forward -> bf16x2 written back IN
//                   PLACE as the next step's A operand; every finished chunk is handed to the
//                   MMA warps and staged through smem per 32-row slab
//      warps 8..11  store warps: copy each staged slab into the CTA's private ring of dpre
//                   images (below) and add its column sums to the layer's bias gradient
//      warps 12,13  MMA issuers, alternating chunks (mlp_issue.cuh): D[128 x 256] = dpre . W
//      warp 14      weight producers: two lanes, alternating W^T operand stages (L2 -> smem
//                   bulk copies)
//      warp 15      ring manager: publishes each finished image (the gpu-scope release fence
//                   waits for the CTA's outstanding stores: ~1-2 k cycles that must not sit in
//                   the store warps' loop)
//  wgrad CTAs (blockIdx >= n_d), weight-stationary: each owns one (layer, input part) job,
//    dW[N_out x K_in] += dpre^T . X accumulated in TENSOR MEMORY over every tile it is dealt
//    (jobs with several CTAs interleave the tiles) and flushed ONCE with fp32 atomics.  Both
//    operands are [samples x features] SWIZZLE_128B images used MN-major: X from the forward
//    stash (HBM, read once), dpre from the ring.  Warps: 0 scout, 1 MMA issuer, 2..5 bulk-copy
//    issuers that also flush the accumulator, 6 releaser; the others are idle.
//
//  The ring replaces round 1's full-size dstash workspace (4.9 KB/sample written by dgrad and
//  read back by wgrad through HBM: 16 GB per C2 step).  Each dgrad CTA owns `depth` 64 KB
//  image slots that it rewrites round-robin (image sequence q = tile iteration * n_img +
//  image index); a slot is consumed by the wgrad CTAs of that layer while it is still in L2,
//  so the dpre images never have to reach HBM.  Flow control is two monotonic counters in
//  global memory: prod[cta] = images completely written by its four store warps (release)
//  and cons[cta][slot] += 2 per image once every reader has landed it in shared memory
//  (images with two readers: += 1 each).  Neither poll sits on a critical path: the store
//  warps fetch the next slot's counter while the current image is still being staged, and a
//  scout warp of each wgrad CTA polls ahead of its bulk-copy issuers.
//
//  Deterministic mode (kDet, fsnerf_mlp_backward_deterministic): the same kernels with every
//  timing-dependent summation order fixed.  dgrad CTA b takes tiles b, b + n_d, ... (no tile
//  counter); each wgrad CTA consumes its tiles in the fixed order (tile iteration, producer) and
//  stores its dW with plain stores into its own workspace slot; the store warps keep private bias
//  sums; the heads kernel writes per-block partials; one reduction kernel then adds every
//  element's partials, in index order, to `grads`.  Every difference sits behind `if constexpr`.
#include "common.cuh"
#include "mlp_common.cuh"
#include "mlp_issue.cuh"

namespace fs {
namespace {

// ------------------------------------------------------------------ dgrad role layout
constexpr int kEpiWarpsB = 8;
constexpr int kRedWarpsB = 4;
constexpr int kWarpRed0 = kEpiWarpsB;                 // 8
constexpr int kWarpMmaB = kEpiWarpsB + kRedWarpsB;    // 12, 13
constexpr int kWarpProdB = kWarpMmaB + kMmaWarps;     // 14
constexpr int kWarpRingB = kWarpProdB + 1;            // 15
constexpr int kThreadsB = (kWarpRingB + 1) * 32;      // 512
constexpr int kImgBars = 32;                          // image-written barriers (>= max ring depth)
constexpr int kStagesB = 4;
constexpr int kSlabBytesB = 32 * 128;
constexpr int kStageBufsB = 3;
constexpr int kMaxLayersB = 12;
constexpr int kImgSlotBytes = 4 * kChunkBytes;        // one ring slot: a [128 x 256] bf16 image

struct SmemB {
  static constexpr int ring = 0;
  static constexpr int staging = ring + kStagesB * kStageBytes;
  static constexpr int bias = staging + 4 * kStageBufsB * kSlabBytesB;   // fp32 [kMaxLayersB][256]
  static constexpr int heads = bias + kMaxLayersB * 256 * 4;             // sigma_w[256], rgb_w[3][128]
  static constexpr int bars = heads + 640 * 4;
  static constexpr int total = bars + 768;
};
struct BarsB {
  static constexpr int w_full = SmemB::bars;
  static constexpr int w_empty = w_full + 8 * kStagesB;
  static constexpr int a_ready = w_empty + 8 * kStagesB;  // [4]
  static constexpr int acc_full = a_ready + 8 * 4;        // [2]
  static constexpr int token = acc_full + 8 * 2;          // [2]
  static constexpr int slab_full = token + 16;            // [4 quarters][kStageBufsB]
  static constexpr int slab_free = slab_full + 8 * 4 * kStageBufsB;
  static constexpr int img_done = slab_free + 8 * 4 * kStageBufsB;   // [kImgBars]
  static constexpr int tmem_slot = img_done + 8 * kImgBars;
  static constexpr int feed = tmem_slot + 8;   // int[5]: tile feed (mlp_issue.cuh: TileSeq)
};
static_assert(BarsB::feed + 32 <= SmemB::total, "barrier block overflows");

struct StepB {
  int target;      // layer whose d(pre-activation) this step produces
  int mask_off;    // stash offset of the 1-bit ReLU mask of the target's forward output, -1: none
  int add_sigma;   // add d(sigma) * w_sigma (target is the last hidden layer)
};
struct PlanB {
  int n_steps;
  int g_branch, branch_mask_off;
  StepB step[kMaxGemm];
};
struct ArgsB {
  long long* trace;
  const uint8_t* packed;
  int64_t n_samples;
  const uint8_t* stash;
  const float* out;
  const float* d_out;
  float* grads;
};
// the dpre image ring shared by the two roles
struct RingB {
  uint32_t* tile_ctr;  // next unclaimed tile (dynamic scheduling of the dgrad CTAs)
  int32_t* tile_of;    // [n_d][row_cap]: tile claimed by dgrad CTA b for its iteration i, -1 past its last
  int row_cap;
  uint8_t* base;    // [n_d][depth] slots of kImgSlotBytes
  uint32_t* prod;   // [n_d]
  uint32_t* cons;   // [n_d][depth]
  int n_d;          // dgrad CTAs
  int depth;        // slots per dgrad CTA
  int n_img;        // images per tile (= GEMM layers)
};

// ------------------------------------------------------------------ wgrad role layout
constexpr int kSlabRows = 64;                     // samples per stage (32: measured 3.40 vs 3.34 ms)
constexpr int kSlabsPerTile = kTileM / kSlabRows;
constexpr int kIssueLanes = 2 * kSlabsPerTile;    // issuing lanes of each of the four producer warps (8 threads per slab)
constexpr int kSlabBytes = kSlabRows * 128;       // 8 KB per 64-feature chunk
// A stage holds one 64-sample slab of the job's operands: (a_chunks + b_chunks) x 8 KB, so the
// small jobs (encoding parts, branch) get a deeper ring out of the same 192 KB: their per-tile
// work is a few hundred cycles and only tiles in flight hide the load latency.
constexpr int kWRingBytes = 24 * 8192;             // 3 stages of a [256 x 256] job
constexpr int kWMaxStages = 8;
constexpr int kWSmemBars = kWRingBytes;            // full[8], empty[8], acc_full, TMEM slot, queue counters
constexpr int kWQueue = 64;                        // tile queue entries (scout -> issuers / releaser)
constexpr int kWSmemQueue = kWSmemBars + 256;
constexpr int kWSmemFlush = kWSmemQueue + kWQueue * 8 + 64;  // two words per queue entry; + per-stage issue clocks (stats)
constexpr int kWSmemTotal = kWSmemFlush + 4 * (32 * 33 * 4);  // + transposition scratch of the four flushing warps
constexpr int kScoutSlots = 5;                     // producers polled per scout lane (32 * 5 >= 148)
constexpr int kMaxJobs = kMaxGemm + 4;

struct WgradJob {
  int a_img, a_chunks;  // dpre image index in the ring sequence, N_out / 64
  int b_off, b_chunks;  // input image (stash record), K_in(part) / 64
  int w_off, ld, col0, ncols, nrows;
  int cta_begin, n_split;
  int cons_inc;         // what this reader adds to cons[] per image (2 / readers of the image)
};
struct WgradPlan {
  int n_jobs, n_ctas;
  WgradJob job[kMaxJobs];
};
// deterministic mode: the partial sums in the caller's workspace (unused by the default kernels)
struct DetB {
  float* wpart;                 // dW of every wgrad CTA: job j's CTA `part` at wpart_off[j] + part * nrows * ncols
  int64_t wpart_off[kMaxJobs];  //   ([nrows x ncols] row-major, floats)
  float* bpart;                 // bias sums [n_d][4 store warps][n_gemm][256]; warp 0's row ends as the CTA's total
  int n_gemm;
};

constexpr int kSmemFused = SmemB::total > kWSmemTotal ? SmemB::total : kWSmemTotal;

// ------------------------------------------------------------------ global flow-control flags
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// The releaser's add needs no release fence: what it orders are the bulk copies' READS of the
// slot, and those have completed when the stage barrier it waited on flipped (a gpu-scope
// release costs ~2.5 k cycles per tile and was the limit of the small wgrad jobs).
__device__ __forceinline__ void red_relaxed_add_u32(uint32_t* p, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// generic-proxy writes to GLOBAL memory made visible by an acquire -> this thread's following
// bulk copies (the all-state-space form costs ~1.3 ms of a 6.8 ms launch here: measured)
__device__ __forceinline__ void fence_proxy_async_global() {
  asm volatile("fence.proxy.async.global;" ::: "memory");
}
// Bounded poll of a monotonic counter (a protocol bug becomes a trap, not a hung box).
__device__ __forceinline__ void wait_counter_ge(const uint32_t* p, uint32_t want, const char* what) {
  uint32_t spins = 0;
  while ((int32_t)(ld_acquire_u32(p) - want) < 0) {
    __nanosleep(64);
    if (++spins > (1u << 22)) {
      printf("fsnerf: %s timeout blk %d thr %d want %u have %u\n", what, blockIdx.x, threadIdx.x, want,
             ld_acquire_u32(p));
      __trap();
    }
  }
}

// Tuning aid (tools/bwd_stats.py): with a trace buffer set, every CTA of the fused launch adds
// the cycles selected warps spend in each wait to trace[kStatBase + 8 * blockIdx + k].
constexpr int kStatBase = 1024;
// ... and the life of the first kEvtImgs images of dgrad CTA 0 as global-timer stamps (ns):
// trace[kEvtBase + kEvtImgs * event + q]
constexpr int kEvtBase = 4096, kEvtImgs = 256;
enum { EVT_SLOT_WAIT = 0, EVT_SLOT_OK, EVT_DONE, EVT_PUB, EVT_SCOUT, EVT_ISSUE, EVT_REL };
__device__ __forceinline__ void evt(long long* trace, int e, uint32_t q) {
  if (trace && q < (uint32_t)kEvtImgs) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    trace[kEvtBase + kEvtImgs * e + q] = (long long)t;
  }
}
struct StatClock {
  long long t;
  bool on;
  __device__ __forceinline__ void start() { if (on) t = clock64(); }
  __device__ __forceinline__ void stop(long long& acc) { if (on) acc += clock64() - t; }
};

// =========================================================================== dgrad role
template <bool kDet>
__device__ __forceinline__ void dgrad_cta(uint8_t* smem, const MlpProgram& prog, const PlanB& plan,
                                          const ArgsB& args, const IssueTable& tab, const RingB& ring,
                                          const DetB& det, const int my_id) {
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // (shuffle: provably warp-uniform)
  const uint32_t bar_w_full = sbase + BarsB::w_full;
  const uint32_t bar_w_empty = sbase + BarsB::w_empty;
  const uint32_t bar_a_ready = sbase + BarsB::a_ready;
  const uint32_t bar_acc_full = sbase + BarsB::acc_full;
  const uint32_t bar_token = sbase + BarsB::token;
  const uint32_t bar_slab_full = sbase + BarsB::slab_full;
  const uint32_t bar_slab_free = sbase + BarsB::slab_free;
  const uint32_t bar_img_done = sbase + BarsB::img_done;
  const uint32_t tmem_slot = sbase + BarsB::tmem_slot;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + BarsB::tmem_slot);
  const float* heads = reinterpret_cast<const float*>(smem + SmemB::heads);
  float* bias_acc = reinterpret_cast<float*>(smem + SmemB::bias);
  const int64_t n_tiles = (args.n_samples + kTileM - 1) / kTileM;
  // Tiles are claimed from a global counter (the ring manager keeps the feed two tiles ahead):
  // the dgrad CTAs do not run at the same speed (they are throttled by different wgrad CTAs and
  // sit at different distances from the L2 slices they stream from), a static split ends with
  // the slowest one.  The deterministic mode takes that cost: CTA b takes tiles b, b + n_d, ...,
  // so that the tiles behind each bias partial and each wgrad CTA's summation order are fixed.
  volatile int* feed = reinterpret_cast<volatile int*>(smem + BarsB::feed);
  const TileSeq seq = kDet ? TileSeq::strided(my_id, ring.n_d, n_tiles) : TileSeq{feed, 0, 0, n_tiles};
  long long* stats = args.trace ? args.trace + kStatBase + 8 * my_id : nullptr;
  const long long t_begin = stats ? clock64() : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStagesB; ++s) {
      mbar_init(bar_w_full + 8 * s, 1);
      mbar_init(bar_w_empty + 8 * s, 1);
    }
    for (int c = 0; c < 4; ++c) mbar_init(bar_a_ready + 8 * c, kEpiWarpsB);
    mbar_init(bar_acc_full, kMmaWarps);
    mbar_init(bar_acc_full + 8, kMmaWarps);
    mbar_init(bar_token, 1);
    mbar_init(bar_token + 8, 1);
    for (int i = 0; i < 4 * kStageBufsB; ++i) {
      mbar_init(bar_slab_full + 8 * i, 2);  // the two epilogue warps of the quarter
      mbar_init(bar_slab_free + 8 * i, 1);  // the quarter's store warp
    }
    for (int i = 0; i < kImgBars; ++i) mbar_init(bar_img_done + 8 * i, kRedWarpsB);
    feed[0] = 0;
    fence_barrier_init();
  }
  if (warp == kWarpMmaB) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < kMaxLayersB * 256; i += kThreadsB) bias_acc[i] = 0.f;
  {  // head weights straight from the packed image's fp32 small-params block (no constant upload)
    const float* __restrict__ small = reinterpret_cast<const float*>(args.packed + prog.small_off);
    for (int i = threadIdx.x; i < 640; i += kThreadsB)
      reinterpret_cast<float*>(smem + SmemB::heads)[i] = __ldg(small + kSmallSigmaW + i);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == kWarpRingB) {
    // ------------------------------------------------ ring manager
    // Image q is complete when the four store warps have arrived on img_done[q % kImgBars]
    // (they run at most `depth` images ahead of this warp, because the slot they would write
    // next is only freed by readers of an image published here).  The arrivals release their
    // stores at CTA scope; the fence below makes the publication cumulative at GPU scope.
    if (lane == 0) {
      uint32_t* my_prod = ring.prod + my_id;
      int32_t* my_tiles = ring.tile_of + (size_t)my_id * ring.row_cap;
      int n_claimed = 0;
      bool dry = false;
      auto claim_upto = [&](int want) {  // tiles of iterations < want are known
        while (n_claimed < want) {
          int t = -1;
          if (!dry && n_claimed < ring.row_cap - 1) {
            if constexpr (kDet) {
              t = (int)seq.get((uint32_t)n_claimed);  // static: the table still tells the scouts
            } else {
              const int64_t c = atomicAdd(ring.tile_ctr, 1u);
              if (c < n_tiles) t = (int)c;
            }
          }
          if (t < 0) dry = true;
          if (n_claimed < ring.row_cap) my_tiles[n_claimed] = t;  // read by the wgrad scouts after they acquire prod
          feed[1 + (n_claimed & 3)] = t;
          __threadfence_block();
          feed[0] = ++n_claimed;
        }
      };
      claim_upto(2);
      uint32_t q = 0;
      for (int it = 0; feed[1 + (it & 3)] >= 0; ++it) {
        claim_upto(it + 3);  // iteration it + 2: the weight producers / MMA issuers run up to ~1 tile ahead
        for (int k = 0; k < ring.n_img; ++k, ++q) {
          mbar_wait_relaxed(bar_img_done + 8 * (q % kImgBars), (q / kImgBars) & 1);
          if (my_id == 0) evt(args.trace, EVT_DONE, q);
          st_release_u32(my_prod, q + 1);  // release = fence.acq_rel.gpu + store
          if (my_id == 0) evt(args.trace, EVT_PUB, q);
        }
      }
      // end marker: the iteration after the last reads as published and its tile_of entry is -1
      st_release_u32(my_prod, q + (uint32_t)ring.n_img);
    }
  } else if (warp == kWarpProdB) {
    IssueBars IB{bar_w_full, bar_w_empty, bar_token, sbase + SmemB::ring};
    if (lane < kProdWarps) producer_loop_thread<kStagesB>(tab, IB, args.packed, seq, lane);
  } else if (warp >= kWarpMmaB) {
    if (tmem_base != 0) __trap();
    IssueBars IB{bar_w_full, bar_w_empty, bar_token, sbase + SmemB::ring};
    issuer_loop<kStagesB>(tab, IB, sbase, seq, (uint32_t)(warp - kWarpMmaB), lane, args.trace);
  } else if (warp >= kWarpRed0) {
    // ------------------------------------------------ store warps: ring images + bias gradients
    // one warp per lane quarter.  Per staged slab (32 rows x 64 features of one chunk): copy it
    // into the current ring image, add its column sums to the layer's bias gradient and free the
    // buffer.  (Summing the columns on the wgrad CTAs, which have every image in shared memory
    // anyway, was measured slower: 4.25 vs 3.42 ms.)
    const int quarter = warp - kWarpRed0;
    const uint32_t stage_base = sbase + SmemB::staging + quarter * (kStageBufsB * kSlabBytesB);
    uint8_t* my_ring = ring.base + (size_t)my_id * ring.depth * kImgSlotBytes;
    uint32_t* my_cons = ring.cons + (size_t)my_id * ring.depth;
    uint32_t n_staged = 0;
    uint32_t q = 0;  // image sequence number of this CTA
    uint32_t cons_seen = 0;  // the upcoming slot's counter, fetched (acquire) one image ahead by lane 0
    StatClock sc{0, stats != nullptr && quarter == 0 && lane == 0};
    long long st_cons = 0, st_slab = 0, st_pub = 0;
    for (uint32_t it = 0; seq.get(it) >= 0; ++it) {
      for (int s = -1; s < plan.n_steps; ++s, ++q) {
        const int layer = (s < 0) ? plan.g_branch : plan.step[s].target;
        const int nchunk = (s < 0) ? 2 : 4;
        const uint32_t slot = q % (uint32_t)ring.depth, gen = q / (uint32_t)ring.depth;
        uint8_t* img = my_ring + (size_t)slot * kImgSlotBytes;
        if (gen > 0) {  // every reader of the slot's previous image has landed it in its smem
          sc.start();
          if (sc.on && my_id == 0) evt(args.trace, EVT_SLOT_WAIT, q);
          if (lane == 0 && (int32_t)(cons_seen - 2u * gen) < 0)
            wait_counter_ge(my_cons + slot, 2u * gen, "dpre ring slot");
          __syncwarp();
          if (sc.on && my_id == 0) evt(args.trace, EVT_SLOT_OK, q);
          sc.stop(st_cons);
        }
        for (int c = 0; c < nchunk; ++c, ++n_staged) {
          const uint32_t b = n_staged % kStageBufsB;
          const uint32_t buf = stage_base + b * kSlabBytesB;
          // deterministic mode: this warp's own running bias sums (two columns per lane) live in
          // the workspace: four private copies in shared memory would take 36 KB, 256 B more than
          // the 227 KB a CTA can have.  Only this lane touches them, so plain loads and stores keep
          // one fixed order; the load is issued before the slab wait to hide its latency.
          float2* bsum = nullptr;
          float2 bprev = make_float2(0.f, 0.f);
          if constexpr (kDet) {
            bsum = reinterpret_cast<float2*>(det.bpart + (((size_t)my_id * 4 + quarter) * det.n_gemm + layer) * 256 +
                                             64 * c) + lane;
            if (it > 0) bprev = *bsum;
          }
          sc.start();
          mbar_wait_relaxed(bar_slab_full + 8 * (quarter * kStageBufsB + b), (n_staged / kStageBufsB) & 1);
          sc.stop(st_slab);
          {
            // coalesced copy with plain loads/stores (512 B per warp instruction): the epilogue
            // then needs no generic->async proxy fence (a MEMBAR.ALL.CTA per chunk) to hand over
            uint4* dst = reinterpret_cast<uint4*>(img + c * kChunkBytes + quarter * kSlabBytesB);
            uint4 t[8];
#pragma unroll
            for (int k = 0; k < 8; ++k)
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(t[k].x), "=r"(t[k].y), "=r"(t[k].z), "=r"(t[k].w)
                           : "r"(buf + (k * 32 + lane) * 16));
#pragma unroll
            for (int k = 0; k < 8; ++k) dst[k * 32 + lane] = t[k];
          }
          {
            float s0 = 0.f, s1 = 0.f, c0 = 0.f, c1 = 0.f;
            const uint8_t* a = smem + SmemB::staging + quarter * (kStageBufsB * kSlabBytesB) + b * kSlabBytesB + ((lane & 3) << 2);
            const uint32_t unit = (uint32_t)lane >> 2;
#pragma unroll
            for (int r = 0; r < 32; r += 2) {
              const uint32_t w0 = *reinterpret_cast<const uint32_t*>(a + r * 128 + ((unit ^ (uint32_t)(r & 7)) << 4));
              const uint32_t w1 = *reinterpret_cast<const uint32_t*>(a + (r + 1) * 128 + ((unit ^ (uint32_t)((r + 1) & 7)) << 4));
              s0 += bf16_lo(w0); s1 += bf16_hi(w0);
              c0 += bf16_lo(w1); c1 += bf16_hi(w1);
            }
            // (a shared-memory float atomic is a CAS loop; four private copies with plain adds
            // measured the same 3.75 ms per launch and cost 36 KB: the store warps are not the limit)
            if constexpr (kDet) {
              *bsum = make_float2(bprev.x + (s0 + c0), bprev.y + (s1 + c1));
            } else {
              atomicAdd(bias_acc + layer * 256 + 64 * c + 2 * lane, s0 + c0);
              atomicAdd(bias_acc + layer * 256 + 64 * c + 2 * lane + 1, s1 + c1);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_slab_free + 8 * (quarter * kStageBufsB + b));
        }
        // this quarter's rows of image q are written (the __syncwarp after the last slab orders
        // every lane's stores before lane 0's arrival): hand the image to the ring manager
        sc.start();
        if (lane == 0) {
          mbar_arrive(bar_img_done + 8 * (q % kImgBars));
          // next image's slot counter: the load's latency hides behind the staging of its first slab
          cons_seen = ld_acquire_u32(my_cons + (q + 1) % (uint32_t)ring.depth);
        }
        sc.stop(st_pub);
      }
    }
    if (sc.on) { stats[1] = st_cons; stats[2] = st_slab; stats[5] = st_pub; }
  } else {
    // ------------------------------------------------ epilogue
    const int quarter = warp & 3, half = warp >> 2;
    const int row = quarter * 32 + lane;
    const uint32_t tmem_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const uint32_t stage_base = sbase + SmemB::staging + quarter * (kStageBufsB * kSlabBytesB);
    uint32_t acc_phase[2] = {0, 0};
    uint32_t n_staged = 0;
    uint32_t titer = 0;
    // stage the 32 bf16 of this thread (16 words) into the quarter's slab and hand it to the
    // store warp (SW128 image: unit u of row r at r*128 + ((u ^ (r&7)) << 4))
    StatClock ec{0, stats != nullptr && threadIdx.x == 0};
    long long st_stage = 0, st_acc = 0;
    auto stage_wait = [&]() {  // the buffer of the upcoming slab has been drained (3 slabs ago)
      const uint32_t b = n_staged % kStageBufsB;
      ec.start();
      mbar_wait(bar_slab_free + 8 * (quarter * kStageBufsB + b), ((n_staged / kStageBufsB) & 1) ^ 1);
      ec.stop(st_stage);
    };
    auto stage_out = [&](const uint32_t (&w)[16]) {
      const uint32_t b = n_staged % kStageBufsB;
      const uint32_t buf = stage_base + b * kSlabBytesB;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        st_shared_v4(buf + lane * 128 + (((uint32_t)(4 * half + j) ^ (uint32_t)(lane & 7)) << 4), w[4 * j],
                     w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_slab_full + 8 * (quarter * kStageBufsB + b));  // release: stores visible
      ++n_staged;
    };
    for (int64_t tile; (tile = seq.get(titer)) >= 0; ++titer) {
      const int64_t p = tile * kTileM + row;
      const bool valid = p < args.n_samples;
      const uint8_t* stash_tile = args.stash + (size_t)tile * prog.stash_tile_bytes;
      // ---- seed: d(out) -> rgb head^T -> d(pre-activation) of the branch layer (128 wide)
      float dz[3] = {0.f, 0.f, 0.f}, dsig = 0.f;
      if (valid) {
        const float4 o4 = __ldg(reinterpret_cast<const float4*>(args.out) + p);
        const float4 g4 = __ldg(reinterpret_cast<const float4*>(args.d_out) + p);
        dz[0] = g4.x * o4.x * (1.0f - o4.x);  // sigmoid'
        dz[1] = g4.y * o4.y * (1.0f - o4.y);
        dz[2] = g4.z * o4.z * (1.0f - o4.z);
        dsig = g4.w;
      }
      {
        // ReLU masks are the 1-bit words the forward wrote (mlp_issue.cuh: relu_bits_*)
        const uint8_t* bm = stash_tile + plan.branch_mask_off;
        uint32_t bw = __ldg(reinterpret_cast<const uint32_t*>(bm + relu_bits_word_off(0, half, row)));
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          const int c0 = 64 * c + 32 * half;
          const uint32_t bw_next =
              (c == 0) ? __ldg(reinterpret_cast<const uint32_t*>(bm + relu_bits_word_off(1, half, row))) : 0u;
          uint32_t w[16];
          const float* wr = heads + 256 + c0;
#pragma unroll
          for (int qq = 0; qq < 16; ++qq) {
            const int i = 2 * qq;
            const float v0 = dz[0] * wr[i] + dz[1] * wr[128 + i] + dz[2] * wr[256 + i];
            const float v1 = dz[0] * wr[i + 1] + dz[1] * wr[128 + i + 1] + dz[2] * wr[256 + i + 1];
            w[qq] = pack_bf16x2(v0, v1) & relu_bits_mask2(bw, qq);
          }
          // step 0 reads its A operand from region 1
          tmem_st16(tmem_lane + 256u + c0, w);
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_a_ready + 8 * c);
          stage_wait();
          stage_out(w);
          bw = bw_next;
        }
      }
      // ---- chain
      for (int s = 0; s < plan.n_steps; ++s) {
        const StepB S = plan.step[s];
        const int r = s & 1;
        const uint32_t region = tmem_lane + (uint32_t)r * 256u + 32u * half;
        const bool last = (s == plan.n_steps - 1);
        const uint8_t* mimg = (S.mask_off >= 0) ? stash_tile + S.mask_off : nullptr;
        const bool add_sigma = S.add_sigma != 0;
        // chunk 0's mask does not depend on the MMAs: fetch it before waiting on the accumulator
        uint32_t mw = mimg ? __ldg(reinterpret_cast<const uint32_t*>(mimg + relu_bits_word_off(0, half, row))) : 0xFFFFFFFFu;
        if (threadIdx.x == 0 && args.trace && my_id == 0 && titer < 4) args.trace[(titer * 16 + s) * 8 + 3] = clock64();
        ec.start();
        mbar_wait(bar_acc_full + 8 * r, acc_phase[r]);
        ec.stop(st_acc);
        acc_phase[r] ^= 1;
        tc_fence_after();
        if (threadIdx.x == 0 && args.trace && my_id == 0 && titer < 4) args.trace[(titer * 16 + s) * 8 + 4] = clock64();
        // The accumulator loads are software-pipelined one chunk ahead through two register
        // buffers: chunk c+1 is in flight from tensor memory while chunk c is converted, masked,
        // written back as the next step's A operand and staged for the ring.
        auto chunk = [&](const int c, uint32_t (&v)[32], uint32_t (&vn)[32]) {
          tmem_ld_wait();  // v = chunk c
          if (c < 3) tmem_ld32(region + 64u * (c + 1), vn);
          const uint32_t mwn = (mimg && c < 3)
                                   ? __ldg(reinterpret_cast<const uint32_t*>(mimg + relu_bits_word_off(c + 1, half, row)))
                                   : 0xFFFFFFFFu;
          uint32_t w[16];
          if (add_sigma) {
            const float* ws = heads + 64 * c + 32 * half;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 w4 = *reinterpret_cast<const float4*>(ws + 4 * i);
              v[4 * i] = __float_as_uint(fmaf(dsig, w4.x, __uint_as_float(v[4 * i])));
              v[4 * i + 1] = __float_as_uint(fmaf(dsig, w4.y, __uint_as_float(v[4 * i + 1])));
              v[4 * i + 2] = __float_as_uint(fmaf(dsig, w4.z, __uint_as_float(v[4 * i + 2])));
              v[4 * i + 3] = __float_as_uint(fmaf(dsig, w4.w, __uint_as_float(v[4 * i + 3])));
            }
          }
#pragma unroll
          for (int qq = 0; qq < 16; ++qq)
            w[qq] = pack_bf16x2(__uint_as_float(v[2 * qq]), __uint_as_float(v[2 * qq + 1])) & relu_bits_mask2(mw, qq);
          if (!last) {
            tmem_st16(region + 64u * c, w);
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_a_ready + 8 * c);
          }
          stage_wait();  // (staging the slab while the tensor-memory store is in flight: within noise, 1-3 %)
          stage_out(w);
          mw = mwn;
        };
        uint32_t va[32], vb[32];
        tmem_ld32(region, va);
#pragma unroll 1
        for (int c = 0; c < 4; c += 2) {
          chunk(c, va, vb);
          chunk(c + 1, vb, va);
        }
        if (threadIdx.x == 0 && args.trace && my_id == 0 && titer < 4) args.trace[(titer * 16 + s) * 8 + 5] = clock64();
      }
    }
    if (ec.on) { stats[3] = st_stage; stats[4] = st_acc; }
  }
  tc_fence_before();
  __syncthreads();
  if (stats && threadIdx.x == 0) stats[0] = clock64() - t_begin;
  if (warp == kWarpMmaB) tmem_dealloc(tmem_base, 512);
  if constexpr (kDet) {
    // the four store warps' sums, combined in warp order into warp 0's row: this CTA's partial
    // (the barrier above made their global stores visible to the whole CTA)
    const size_t wstride = (size_t)det.n_gemm * 256;
    float* mine = det.bpart + (size_t)my_id * 4 * wstride;
    for (int g = 0; g < prog.n_gemm; ++g) {
      const int ncols = prog.layer[g].n_halves * 128;
      if ((int)threadIdx.x < ncols) {
        float* p = mine + g * 256 + threadIdx.x;
        p[0] = ((p[0] + p[wstride]) + p[2 * wstride]) + p[3 * wstride];
      }
    }
  } else {
    for (int g = 0; g < prog.n_gemm; ++g) {  // bias gradients of this CTA -> global
      const int ncols = prog.layer[g].n_halves * 128;
      if ((int)threadIdx.x < ncols)
        atomicAdd(args.grads + prog.layer[g].bias_off + threadIdx.x, bias_acc[g * 256 + threadIdx.x]);
    }
  }
}

// =========================================================================== wgrad role
template <bool kDet>
__device__ __forceinline__ void wgrad_cta(uint8_t* smem, const MlpProgram& prog, const ArgsB& args,
                                          const WgradPlan& plan, const RingB& ring, const DetB& det,
                                          const int cta) {
  const uint32_t sbase = smem_u32(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // (shuffle: provably warp-uniform)
  const uint32_t bar_full = sbase + kWSmemBars;
  const uint32_t bar_empty = bar_full + 8 * kWMaxStages;
  const uint32_t bar_acc_full = bar_empty + 8 * kWMaxStages;
  const uint32_t tmem_slot = bar_acc_full + 8;
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem + kWSmemBars + 8 * (2 * kWMaxStages + 1));
  // The scout appends every tile whose dpre image is published to a queue in shared memory
  // (ready_upto entries so far); released_upto = entries the releaser is done with.
  volatile uint32_t* ready_upto = reinterpret_cast<volatile uint32_t*>(smem + kWSmemBars + 160);
  volatile uint32_t* released_upto = reinterpret_cast<volatile uint32_t*>(smem + kWSmemBars + 164);
  volatile uint32_t* queue = reinterpret_cast<volatile uint32_t*>(smem + kWSmemQueue);
  int j = 0;
  while (j + 1 < plan.n_jobs && cta >= plan.job[j + 1].cta_begin) ++j;
  const WgradJob& J = plan.job[j];
  const int part = cta - J.cta_begin;
  // This CTA reads the images of dgrad CTAs part, part + n_split, ... (every tile of theirs), in
  // whatever order they are published: a consumer bound to a fixed tile order would stall on one
  // late producer while the others fill their rings and stall too.
  const int n_mine = (ring.n_d > part) ? (ring.n_d - part + J.n_split - 1) / J.n_split : 0;
  // how many tiles that is is only known at the end (the dgrad CTAs claim tiles dynamically): the
  // scout publishes the total once every producer has sent its end marker
  volatile uint32_t* final_count = reinterpret_cast<volatile uint32_t*>(smem + kWSmemBars + 168);
  auto have_tile = [&](uint32_t n) -> bool {  // false: no n-th tile, the CTA's list has ended
    uint32_t spins = 0;
    while (*ready_upto <= n) {
      if (*final_count != 0xFFFFFFFFu) return n < *final_count;
      __nanosleep(32);
      if (++spins > (1u << 24)) { printf("fsnerf: wgrad scout timeout blk %d thr %d\n", blockIdx.x, threadIdx.x); __trap(); }
    }
    __threadfence_block();
    return true;
  };
  long long* stats = args.trace ? args.trace + kStatBase + 8 * (ring.n_d + cta) : nullptr;
  const long long t_begin = stats ? clock64() : 0;
  const int n_cp = J.a_chunks + J.b_chunks;  // operand chunks per stage
  const uint32_t stage_bytes = (uint32_t)n_cp * kSlabBytes;
  volatile long long* issue_clk = reinterpret_cast<volatile long long*>(smem + kWSmemQueue + kWQueue * 8);  // stats only
  const uint32_t n_stages = (kWRingBytes / stage_bytes) < (uint32_t)kWMaxStages ? (kWRingBytes / stage_bytes) : (uint32_t)kWMaxStages;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kWMaxStages; ++s) {
      mbar_init(bar_full + 8 * s, 8);   // the eight issuing threads of a slab (four lanes of two producer warps)
      mbar_init(bar_empty + 8 * s, 2);  // MMA commit + releaser
    }
    mbar_init(bar_acc_full, 1);
    *ready_upto = 0;
    *released_upto = 0;
    *final_count = (n_mine > 0) ? 0xFFFFFFFFu : 0u;
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const int n_mh = J.a_chunks / 2;

  {
    if (warp >= 2 && warp < 6) {
      // four producer warps (the epilogue warps, idle during the main loop): bulk copies issued
      // by one thread do not overlap (~440 cycles each, tools/l2_bench.cu), so a tile's slab copies
      // (8 KB each: 64 rows of one chunk image) are spread over SIXTEEN issuing threads — lanes
      // 0..3 of warps 2, 3 take the tile's first slab, those of warps 4, 5 its second — each arming
      // its stage's barrier for its own bytes: at most one or two copies per thread and tile.
      const int pw = (warp - 2) * kIssueLanes + lane;  // issuing thread index (lanes 0..kIssueLanes-1 issue)
      const int my_slab = ((warp - 2) * kIssueLanes) >> 3, my_c = pw & 7;  // (one slab per warp or per warp pair)
      uint32_t fenced_upto = 0;
      StatClock pc{0, stats != nullptr && warp == 2 && lane == 0};
      long long st_ready = 0, st_empty = 0;
      for (uint32_t n = 0;; ++n) {
        pc.start();
        if (!have_tile(n)) break;  // (every lane: the warp stays together)
        pc.stop(st_ready);
        const uint32_t cnt = (uint32_t)kSlabsPerTile * n + (uint32_t)my_slab;
        const uint32_t stage = cnt % n_stages, phase = (cnt / n_stages) & 1;
        pc.start();
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        pc.stop(st_empty);
        if (lane < kIssueLanes) {
          if (n >= fenced_upto) {
            // one generic -> async proxy fence covers every tile the scout has published so far
            const uint32_t r = *ready_upto;
            __threadfence_block();
            fence_proxy_async_global();
            fenced_upto = r;
          }
          const int64_t tile = queue[2 * (n % kWQueue)];
          const uint32_t bi = queue[2 * (n % kWQueue) + 1];  // producer | its iteration << 8
          const int b = (int)(bi & 255u);
          const uint32_t q = (bi >> 8) * (uint32_t)ring.n_img + (uint32_t)J.a_img;
          const uint8_t* a_img = ring.base + ((size_t)b * ring.depth + q % (uint32_t)ring.depth) * kImgSlotBytes;
          const uint8_t* b_img = args.stash + (size_t)tile * prog.stash_tile_bytes + J.b_off;
          if (b == 0 && pw == 0 && J.cons_inc == 2) evt(args.trace, EVT_ISSUE, q);
          const uint32_t sa = sbase + stage * stage_bytes, sb = sa + (uint32_t)J.a_chunks * kSlabBytes;
          int mine = 0;
          for (int c = my_c; c < n_cp; c += 8) ++mine;
          if (my_c == 0 && stats) issue_clk[stage] = clock64();
          mbar_arrive_expect_tx(bar_full + 8 * stage, (uint32_t)mine * kSlabBytes);
          // (L2 eviction hints — evict_first on the stash stream, evict_last on the ring reads and
          // writes — recover the 10-slot ring's loss against the 5-slot one, 4.00 -> 3.75 ms, and
          // add nothing to the 5-slot ring: it is resident without them)
          for (int c = my_c; c < n_cp; c += 8) {
            if (c < J.a_chunks)
              bulk_g2s(sa + c * kSlabBytes, a_img + c * kChunkBytes + my_slab * kSlabBytes, kSlabBytes,
                       bar_full + 8 * stage);
            else
              bulk_g2s(sb + (c - J.a_chunks) * kSlabBytes, b_img + (c - J.a_chunks) * kChunkBytes + my_slab * kSlabBytes,
                       kSlabBytes, bar_full + 8 * stage);
          }
        }
        __syncwarp();
      }
      if (pc.on) { stats[1] = st_ready; stats[2] = st_empty; }
    } else if (warp == 6) {
      // releaser: once the last slab of a tile has landed, the whole dpre image is in shared
      // memory and its ring slot goes back to the dgrad CTA.  It also arrives on the stage's
      // empty barrier so that it can never fall a barrier phase behind.
      if (lane == 0) {
        uint32_t cnt = 0;
        for (uint32_t n = 0; have_tile(n); ++n) {
          for (int slab = 0; slab < kTileM / kSlabRows; ++slab, ++cnt) {
            const uint32_t stage = cnt % n_stages, phase = (cnt / n_stages) & 1;
            mbar_wait_relaxed(bar_full + 8 * stage, phase);
            if (slab == kTileM / kSlabRows - 1) {
              const uint32_t bi = queue[2 * (n % kWQueue) + 1];
              const int b = (int)(bi & 255u);
              const uint32_t q = (bi >> 8) * (uint32_t)ring.n_img + (uint32_t)J.a_img;
              red_relaxed_add_u32(ring.cons + (size_t)b * ring.depth + q % (uint32_t)ring.depth, (uint32_t)J.cons_inc);
              *released_upto = (uint32_t)(n + 1);
              if (b == 0 && J.cons_inc == 2) evt(args.trace, EVT_REL, q);
            }
            mbar_arrive(bar_empty + 8 * stage);
          }
        }
      }
    } else if (warp == 0 && kDet) {
      // deterministic scout: the queue takes this CTA's tiles in the fixed order (tile iteration,
      // producer index), waiting for the next one in that order even when others are ready, so the
      // MMA warp adds them into tensor memory in a fixed sequence.  Lane l watches the l-th entry
      // not yet queued; the ready prefix is appended.
      //   No deadlock: every consumer follows the same global order and every producer writes its
      // images in order.  Take the smallest (iteration, producer) pair not fully consumed.  Each of
      // its readers has consumed everything smaller, so it waits for this pair and nothing else.
      // The producer's first image of the pair needs a slot freed by an image of an earlier
      // iteration (all consumed); image k of the pair needs the slot of image k - depth, an
      // earlier image of the same pair or of an earlier iteration, which its readers can land as
      // soon as it is published.  So the pair completes, and by induction every pair does.
      //   Watchdogs: the longest wait here is one producer's next image (at most one launch's
      // length, milliseconds); the bounds below, like the dgrad side's slot wait, are ~0.3 s or more
      // of no progress.
      const int64_t n_tiles = (args.n_samples + kTileM - 1) / kTileM;
      uint32_t enq = 0, idle = 0;
      for (uint32_t it = 0;; ++it) {
        // producers of this CTA with a tile in iteration it: b = part + k n_split with
        // b + it n_d < n_tiles (static tiles), a prefix k < K of the list since b grows with k
        const int64_t left = n_tiles - (int64_t)it * ring.n_d - part;
        int K = left <= 0 ? 0 : (int)((left + J.n_split - 1) / J.n_split);
        if (K > n_mine) K = n_mine;
        if (K <= 0) break;
        const uint32_t need = it * (uint32_t)ring.n_img + (uint32_t)J.a_img + 1u;
        for (int k0 = 0; k0 < K; k0 += 32) {
          const int cnt = (K - k0 < 32) ? K - k0 : 32;
          const int b = part + (k0 + lane) * J.n_split;
          bool ready = lane >= cnt;
          int32_t t = -1;
          for (int done = 0; done < cnt;) {
            if (!ready && (int32_t)(ld_acquire_u32(ring.prod + b) - need) >= 0) {
              t = ring.tile_of[(size_t)b * ring.row_cap + it];
              if (t < 0) { printf("fsnerf: wgrad scout: no tile, blk %d producer %d iteration %u\n", blockIdx.x, b, it); __trap(); }
              ready = true;
            }
            const uint32_t nready = ~__ballot_sync(0xffffffffu, ready);
            const int upto = nready ? __ffs(nready) - 1 : 32;  // lanes below `upto` are all ready
            const int n_new = (upto < cnt ? upto : cnt) - done;
            if (n_new > 0) {
              if (lane == 0) {  // room in the queue
                uint32_t spins = 0;
                while ((int32_t)(enq + (uint32_t)n_new - *released_upto) > kWQueue) {
                  __nanosleep(64);
                  if (++spins > (1u << 24)) { printf("fsnerf: wgrad queue timeout blk %d\n", blockIdx.x); __trap(); }
                }
              }
              __syncwarp();
              if (lane >= done && lane < done + n_new) {
                const uint32_t pos = enq + (uint32_t)(lane - done);
                queue[2 * (pos % kWQueue)] = (uint32_t)t;
                queue[2 * (pos % kWQueue) + 1] = (uint32_t)b | (it << 8);
              }
              enq += (uint32_t)n_new;
              done += n_new;
              __syncwarp();
              if (lane == 0) {
                __threadfence_block();
                *ready_upto = enq;
              }
              idle = 0;
            } else {
              __nanosleep(128);
              if (++idle > (1u << 22)) {
                if (lane == 0) printf("fsnerf: wgrad scout waited too long for producer %d, blk %d enq %u\n",
                                      part + (k0 + done) * J.n_split, blockIdx.x, enq);
                __trap();
              }
            }
          }
        }
      }
      if (lane == 0) {
        __threadfence_block();
        *final_count = enq;
      }
    } else if (warp == 0) {
      // scout: every lane watches up to kScoutSlots of this CTA's producers and appends a tile to
      // the queue as soon as its image is published (at most one per producer per sweep)
      uint32_t nxt[kScoutSlots];   // next iteration of each watched producer, 0xFFFFFFFF: it has ended
#pragma unroll
      for (int sl = 0; sl < kScoutSlots; ++sl) nxt[sl] = (lane + 32 * sl < n_mine) ? 0u : 0xFFFFFFFFu;
      uint32_t enq = 0, idle = 0;
      for (;;) {
        bool any = false, live = false;
#pragma unroll
        for (int sl = 0; sl < kScoutSlots; ++sl) {
          const int k = lane + 32 * sl;
          const int b = part + k * J.n_split;
          bool flag = false;
          int32_t t = -1;
          if (nxt[sl] != 0xFFFFFFFFu) {
            const uint32_t need = nxt[sl] * (uint32_t)ring.n_img + (uint32_t)J.a_img + 1u;
            if ((int32_t)(ld_acquire_u32(ring.prod + b) - need) >= 0) {
              t = ring.tile_of[(size_t)b * ring.row_cap + nxt[sl]];
              if (t < 0) nxt[sl] = 0xFFFFFFFFu;  // end marker
              else flag = true;
            }
          }
          live = live || nxt[sl] != 0xFFFFFFFFu;
          const uint32_t mask = __ballot_sync(0xffffffffu, flag);
          if (mask) {
            const uint32_t cntm = __popc(mask);
            if (lane == 0) {  // room in the queue
              uint32_t spins = 0;
              while ((int32_t)(enq + cntm - *released_upto) > kWQueue) {
                __nanosleep(64);
                if (++spins > (1u << 24)) { printf("fsnerf: wgrad queue timeout blk %d\n", blockIdx.x); __trap(); }
              }
            }
            __syncwarp();
            if (flag) {
              const uint32_t pos = enq + __popc(mask & ((1u << lane) - 1u));
              queue[2 * (pos % kWQueue)] = (uint32_t)t;
              queue[2 * (pos % kWQueue) + 1] = (uint32_t)b | (nxt[sl] << 8);
              if (b == 0) evt(args.trace, EVT_SCOUT, nxt[sl] * (uint32_t)ring.n_img + (uint32_t)J.a_img);
              ++nxt[sl];
            }
            enq += cntm;
            __syncwarp();
            if (lane == 0) {
              __threadfence_block();
              *ready_upto = enq;
            }
            any = true;
          }
        }
        if (!__any_sync(0xffffffffu, live)) break;
        if (any) {
          idle = 0;
        } else {
          __nanosleep(128);
          if (++idle > (1u << 22)) {
            if (lane == 0) printf("fsnerf: wgrad scout found nothing to do for too long, blk %d enq %u\n", blockIdx.x, enq);
            __trap();
          }
        }
      }
      if (lane == 0) {
        __threadfence_block();
        *final_count = enq;
      }
    } else if (warp == 1) {
      // A = dpre^T (M = output features), B = X^T (N = input features); both MN-major:
      // 64-feature groups LBO = kSlabBytes apart, 8-sample K groups SBO = 1024 B apart.
      const uint32_t idesc = umma_idesc_bf16(128, J.b_chunks * 64, 1, 1);
      uint32_t cnt = 0;
      StatClock mc{0, stats != nullptr && lane == 0};
      long long st_full = 0, st_lat = 0;
      uint32_t n_done = 0;
      for (uint32_t n = 0; have_tile(n); ++n, ++n_done) {
        for (int slab = 0; slab < kTileM / kSlabRows; ++slab, ++cnt) {
          const uint32_t stage = cnt % n_stages, phase = (cnt / n_stages) & 1;
          mc.start();
          mbar_wait(bar_full + 8 * stage, phase);
          mc.stop(st_full);
          if (mc.on) st_lat += clock64() - issue_clk[stage];
          tc_fence_after();
          if (elect_one()) {  // (elected, not `lane == 0`: the compiler then knows one thread issues)
            const uint32_t sa = sbase + stage * stage_bytes, sb = sa + (uint32_t)J.a_chunks * kSlabBytes;
            for (int mh = 0; mh < n_mh; ++mh) {
#pragma unroll
              for (int ks = 0; ks < kSlabRows / 16; ++ks) {
                umma_bf16_ss(tmem_base + mh * 256,
                             umma_desc_sw128(sa + mh * 2 * kSlabBytes + ks * 2048, kSlabBytes, 1024),
                             umma_desc_sw128(sb + ks * 2048, kSlabBytes, 1024), idesc,
                             (cnt > 0 || ks > 0) ? 1u : 0u);
              }
            }
            umma_commit(bar_empty + 8 * stage);
          }
          __syncwarp();
        }
      }
      if (elect_one()) umma_commit(bar_acc_full);  // the same thread every time: it issued the MMAs
      __syncwarp();
      if (mc.on) { stats[3] = st_full; stats[4] = n_done; stats[6] = j; stats[5] = st_lat; }
    }
    if (warp >= 2 && warp < 6 && (kDet || *final_count != 0)) {
      const int quarter = warp & 3;
      mbar_wait(bar_acc_full, 0);
      tc_fence_after();
      // deterministic mode: plain stores into this CTA's own slot (zeros if it was dealt no tile)
      float* slot = nullptr;
      bool none = false;
      if constexpr (kDet) {
        slot = det.wpart + det.wpart_off[j] + (int64_t)part * J.nrows * J.ncols;
        none = *final_count == 0;
      }
      // The accumulator tile of a warp is [32 rows (lanes) x 32 columns (registers)]; a straight
      // flush would issue atomics strided by a weight row (32 cache lines per instruction).  It is
      // transposed through shared memory instead: lane = column, one line per atomic.
      float* tr = reinterpret_cast<float*>(smem + kWSmemFlush + (warp - 2) * (32 * 33 * 4));
      for (int mh = 0; mh < n_mh; ++mh) {
        const int rbase = mh * 128 + quarter * 32;
        for (int c0 = 0; c0 < J.b_chunks * 64; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + mh * 256 + c0, v);
          tmem_ld_wait();
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 32; ++i) tr[lane * 33 + i] = __uint_as_float(v[i]);
          __syncwarp();
          if (c0 + lane < J.ncols) {
            if constexpr (kDet) {
              float* __restrict__ pcol = slot + c0 + lane;
#pragma unroll 8
              for (int rr = 0; rr < 32; ++rr)
                if (rbase + rr < J.nrows) pcol[(size_t)(rbase + rr) * J.ncols] = none ? 0.f : tr[rr * 33 + lane];
            } else {
              float* __restrict__ gcol = args.grads + J.w_off + J.col0 + c0 + lane;
#pragma unroll 8
              for (int rr = 0; rr < 32; ++rr)
                if (rbase + rr < J.nrows) atomicAdd(gcol + (size_t)(rbase + rr) * J.ld, tr[rr * 33 + lane]);
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (stats && threadIdx.x == 0) stats[0] = clock64() - t_begin;
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

template <bool kDet>
__global__ void __launch_bounds__(kThreadsB, 1)
mlp_bwd_fused_kernel(const __grid_constant__ MlpProgram prog, const __grid_constant__ PlanB plan,
                     const __grid_constant__ ArgsB args, const __grid_constant__ IssueTable tab,
                     const __grid_constant__ WgradPlan wplan, const __grid_constant__ RingB ring,
                     const __grid_constant__ DetB det) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  // Roles by contiguous block ranges.  Consecutive block indices land on the two SMs of one TPC
  // (measured: blockIdx 2k, 2k+1 -> smid 2j, 2j+1), so with an even n_d both SMs of a TPC run the
  // SAME role.  Interleaving the roles (one dgrad + one wgrad CTA per TPC, to spread the wgrad
  // role's ~2.5x heavier L2 ingest) was measured much SLOWER: 5.65 vs 3.76 ms per C2 launch on the
  // same box, some wgrad CTAs then see 6-8 k cycles per stage copy instead of 3-4 k.
  const int b = (int)blockIdx.x;
  const bool is_d = b < ring.n_d;
  const int id = is_d ? b : b - ring.n_d;
  const int lin = is_d ? id : ring.n_d + id;  // index of this CTA's tuning records
  if (args.trace && threadIdx.x == 0) {  // tuning aid: CTA life span on the global timer (ns)
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    args.trace[6144 + 2 * lin] = (long long)t;
    uint32_t smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    args.trace[6500 + lin] = (long long)smid;
  }
  if (is_d)
    dgrad_cta<kDet>(smem, prog, plan, args, tab, ring, det, id);
  else
    wgrad_cta<kDet>(smem, prog, args, wplan, ring, det, id);
  if (args.trace && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    args.trace[6144 + 2 * lin + 1] = (long long)t;
  }
}

// =========================================================================== heads (SIMT)
struct HeadsArgs {
  const uint8_t* stash;
  int stash_tile_bytes;
  int h_off;   // stash offset of the last hidden layer's output image (sigma head input)
  int hb_off;  // stash offset of the branch output image (rgb head input)
  int64_t n_samples, n_tiles;
  const float* out;
  const float* d_out;
  float* g_sigma_w; float* g_sigma_b; float* g_rgb_w; float* g_rgb_b;
};

__device__ __forceinline__ uint4 ldg_u4(const void* p) {
  return __ldg(reinterpret_cast<const uint4*>(p));
}

// 256 threads: thread t owns 16-byte unit (t & 31) [= 8 features of chunk (t&31)>>3]
// of the 256-wide h image and, if (t & 31) < 16, of the 128-wide hb image; the 8
// row-groups (t >> 5) split the 128 rows.  Every load is a coalesced 16 B / lane.
// kDet: no atomics; block b writes its sums to part[b * kHeadPart + ...] (kHeadPart layout below).
constexpr int kHeadPart = 648;  // sigma_w [256], rgb_w [3][128], rgb_b [3], sigma_b, padding
template <bool kDet>
__global__ void __launch_bounds__(256, 3)
mlp_heads_wgrad_kernel(const __grid_constant__ HeadsArgs a, float* __restrict__ part) {
  __shared__ float4 dsm[kTileM];  // (dz0, dz1, dz2, dsigma) per row
  __shared__ float red[8][32][33];
  const int t = threadIdx.x, u = t & 31, rg = t >> 5;
  const int chunk = u >> 3, unit = u & 7;
  float acc_s[8], acc_r[3][8];
  float4 acc_b = make_float4(0.f, 0.f, 0.f, 0.f);  // bias sums: lane 0 of each row group
#pragma unroll
  for (int e = 0; e < 8; ++e) { acc_s[e] = 0.f; acc_r[0][e] = acc_r[1][e] = acc_r[2][e] = 0.f; }
  // (dz, dsigma) of this thread's row of the NEXT tile, fetched one tile ahead so that its
  // latency overlaps the current tile's streaming loop
  auto load_d = [&](int64_t tile) {
    float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t p = tile * kTileM + t;
    if (t < kTileM && tile < a.n_tiles && p < a.n_samples) {
      const float4 o4 = __ldg(reinterpret_cast<const float4*>(a.out) + p);
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(a.d_out) + p);
      d = make_float4(g4.x * o4.x * (1.f - o4.x), g4.y * o4.y * (1.f - o4.y),
                      g4.z * o4.z * (1.f - o4.z), g4.w);
    }
    return d;
  };
  float4 d_next = load_d(blockIdx.x);
  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    __syncthreads();
    if (t < kTileM) dsm[t] = d_next;
    __syncthreads();
    d_next = load_d(tile + gridDim.x);
    const uint8_t* rec = a.stash + (size_t)tile * a.stash_tile_bytes;
    const uint8_t* h = rec + a.h_off + chunk * kChunkBytes;
    // lanes with u >= 16 have no hb column: they re-read a valid unit (same cache lines as
    // lanes 0..15) and their rgb partial sums are never used, so the loop stays branch-free
    // and every load of a batch is in flight before the first use
    const uint8_t* hb = rec + a.hb_off + (chunk & 1) * kChunkBytes;
    constexpr int kBatch = 4;
#pragma unroll 1
    for (int r0 = 0; r0 < kTileM / 8; r0 += kBatch) {
      uint4 hv[kBatch], bv[kBatch];
#pragma unroll
      for (int k = 0; k < kBatch; ++k) {
        const int r = rg * (kTileM / 8) + r0 + k;
        const uint32_t off = sw128_off(r, unit);
        hv[k] = ldg_u4(h + off);
        bv[k] = ldg_u4(hb + off);
      }
#pragma unroll
      for (int k = 0; k < kBatch; ++k) {
        const int r = rg * (kTileM / 8) + r0 + k;
        const float4 d = dsm[r];
        if (u == 0) { acc_b.x += d.x; acc_b.y += d.y; acc_b.z += d.z; acc_b.w += d.w; }
        const uint32_t hw[4] = {hv[k].x, hv[k].y, hv[k].z, hv[k].w};
        const uint32_t bw[4] = {bv[k].x, bv[k].y, bv[k].z, bv[k].w};
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
          acc_s[2 * qq] = fmaf(d.w, bf16_lo(hw[qq]), acc_s[2 * qq]);
          acc_s[2 * qq + 1] = fmaf(d.w, bf16_hi(hw[qq]), acc_s[2 * qq + 1]);
          const float x0 = bf16_lo(bw[qq]), x1 = bf16_hi(bw[qq]);
          acc_r[0][2 * qq] = fmaf(d.x, x0, acc_r[0][2 * qq]); acc_r[0][2 * qq + 1] = fmaf(d.x, x1, acc_r[0][2 * qq + 1]);
          acc_r[1][2 * qq] = fmaf(d.y, x0, acc_r[1][2 * qq]); acc_r[1][2 * qq + 1] = fmaf(d.y, x1, acc_r[1][2 * qq + 1]);
          acc_r[2][2 * qq] = fmaf(d.z, x0, acc_r[2][2 * qq]); acc_r[2][2 * qq + 1] = fmaf(d.z, x1, acc_r[2][2 * qq + 1]);
        }
      }
    }
  }
  // combine the 8 row-groups through shared memory, then one atomic per feature
  __syncthreads();
#pragma unroll
  for (int e = 0; e < 8; ++e) red[rg][u][e] = acc_s[e];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int e = 0; e < 8; ++e) red[rg][u][8 + 8 * c + e] = acc_r[c][e];
  if constexpr (kDet) {
    if (u == 0) dsm[rg] = acc_b;  // (dsm is free: its last reader passed the barrier above)
  }
  __syncthreads();
  float* my = nullptr;
  if constexpr (kDet) my = part + (size_t)blockIdx.x * kHeadPart;
  {
    // thread t -> feature t of h (sigma head): unit t>>3, element t&7
    float s = 0.f;
    for (int g = 0; g < 8; ++g) s += red[g][t >> 3][t & 7];
    if constexpr (kDet) my[t] = s; else atomicAdd(a.g_sigma_w + t, s);
    if (t < 128) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float r3 = 0.f;
        for (int g = 0; g < 8; ++g) r3 += red[g][t >> 3][8 + 8 * c + (t & 7)];
        if constexpr (kDet) my[256 + c * 128 + t] = r3; else atomicAdd(a.g_rgb_w + c * 128 + t, r3);
      }
    }
  }
  if constexpr (kDet) {
    if (t == 0) {  // the row groups' bias sums in row-group order
      float4 bs = dsm[0];
      for (int g = 1; g < 8; ++g) {
        const float4 d = dsm[g];
        bs.x += d.x; bs.y += d.y; bs.z += d.z; bs.w += d.w;
      }
      my[640] = bs.x; my[641] = bs.y; my[642] = bs.z; my[643] = bs.w;
    }
  } else if (u == 0) {
    atomicAdd(a.g_rgb_b + 0, acc_b.x);
    atomicAdd(a.g_rgb_b + 1, acc_b.y);
    atomicAdd(a.g_rgb_b + 2, acc_b.z);
    atomicAdd(a.g_sigma_b, acc_b.w);
  }
}

// =========================================================================== deterministic reduction
// grads[i] = grads[i] + (sum of element i's partials in index order): the wgrad CTAs of its job,
// the dgrad CTAs (biases) or the heads blocks.  One thread per element, so the order is fixed.
struct RedSeg {
  int64_t dst;          // float offset in grads of element (0, 0)
  int64_t src;          // float offset in the partials of part 0's element (0, 0)
  int64_t part_stride;  // floats between consecutive parts
  int rows, cols, dst_ld, src_ld, n_parts;
};
constexpr int kMaxRedSegs = kMaxJobs + kMaxLayersB + 4;
struct RedPlan {
  int n;
  RedSeg seg[kMaxRedSegs];
};
__global__ void __launch_bounds__(256)
mlp_bwd_det_reduce_kernel(const __grid_constant__ RedPlan plan, const float* __restrict__ parts,
                          float* __restrict__ grads) {
  const RedSeg& S = plan.seg[blockIdx.y];
  const int64_t n = (int64_t)S.rows * S.cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / S.cols, c = i % S.cols;
    const float* p = parts + S.src + r * S.src_ld + c;
    float s = p[0];
    for (int k = 1; k < S.n_parts; ++k) s += p[(int64_t)k * S.part_stride];
    float* g = grads + S.dst + r * S.dst_ld + c;
    *g = *g + s;
  }
}

// ------------------------------------------------------------------ host-side plan
constexpr int kFlagBytes = 32768;  // prod [148] + cons [148][kMaxRingDepth] uint32, padded
constexpr int kMaxRingDepth = 32;
// CTAs of the fused launch that take the weight-gradient role: swept 54-62, all within 2 % (56 was
// 1-2 % ahead of 58 on a fast box and behind on a slow one; profiles/README.md)
constexpr int kWgradCtas = 58;
// per-tile overhead of a wgrad job in the job cost model (see the cost comment in fsnerf_mlp_backward)
constexpr int kJobOverheadCycles = 3000;
// tile_of rows: a dgrad CTA may claim up to 4x its even share (then it stops claiming)
int tile_row_cap(int64_t n_tiles, int n_d) { return (int)(4 * ((n_tiles + n_d - 1) / n_d) + 8); }
int64_t tile_table_bytes(int64_t n_tiles, int n_d) {
  return (((int64_t)n_d * tile_row_cap(n_tiles, n_d) * 4) + 1023) & ~(int64_t)1023;
}
int ring_depth_for(int n_img) {
  // half a tile's images.  The slots are rewritten every few microseconds and must stay in L2
  // against the stash and weight streams passing through it: measured 3.75 ms (5 slots, 29 MB for
  // 90 dgrad CTAs) vs 4.06 ms (10 slots) vs 4.2 ms (20 slots) per C2 fused launch on the same box;
  // below 4 the producers stall on their readers (2 slots: 4.04 ms)
  int d = (n_img + 1) / 2;
  if (d < 2) d = 2;
  if (d > kMaxRingDepth) d = kMaxRingDepth;
  return d;
}

struct SplitB {
  int n_d, n_w;
};
// how the (at most) 148 CTAs of the fused launch divide into the two roles
SplitB split_roles(int n_jobs, int64_t n_tiles) {
  SplitB s;
  int n_w = kWgradCtas;
  if (n_w < n_jobs) n_w = n_jobs;
  if (n_w > kNumSMs - 1) n_w = kNumSMs - 1;
  // a job never gets more CTAs than there are tiles
  if ((int64_t)n_w > n_tiles * n_jobs) n_w = (int)(n_tiles * n_jobs);
  int n_d = kNumSMs - n_w;
  if ((int64_t)n_d > n_tiles) n_d = (int)n_tiles;
  s.n_d = n_d;
  s.n_w = n_w;
  return s;
}

int count_jobs(const MlpProgram& P) {
  int n = 0;
  for (int g = 0; g < P.n_gemm; ++g) n += (P.layer[g].n_act_chunks ? 1 : 0) + (P.layer[g].use_aux ? 1 : 0);
  return n;
}

int heads_grid(int64_t n_tiles) {
  // one resident wave (3 CTAs per SM): 0.203 vs 0.218 ms per C2 step with two waves, 0.237 with three.
  // (On the wgrad CTAs' idle warps the heads cost ~4800 CUDA-core cycles per tile, more than the
  // jobs that stage their inputs can absorb: measured 6.4-9.4 ms per launch against 0.22 ms here.)
  return (int)(n_tiles < 3 * kNumSMs ? n_tiles : 3 * kNumSMs);
}

// ---- wgrad plan: (layer, input part) jobs, CTAs split in proportion to their cycles per tile
int build_wgrad_plan(const MlpProgram& P, int64_t n_tiles, WgradPlan& WP, SplitB& sp) {
  WP.n_jobs = 0;
  double cost[kMaxJobs], total = 0;
  int readers[kMaxGemm];
  for (int g = 0; g < P.n_gemm; ++g) readers[g] = (P.layer[g].n_act_chunks ? 1 : 0) + (P.layer[g].use_aux ? 1 : 0);
  for (int g = 0; g < P.n_gemm; ++g) {
    const GemmLayer& L = P.layer[g];
    const int a_chunks = L.n_halves * 2;
    for (int part = 0; part < 2; ++part) {
      if (part == 0 && L.n_act_chunks == 0) continue;
      if (part == 1 && !L.use_aux) continue;
      FS_REQUIRE(WP.n_jobs < kMaxJobs, "mlp_backward: too many wgrad jobs");
      WgradJob& J = WP.job[WP.n_jobs];
      J.a_img = P.n_gemm - 1 - g; J.a_chunks = a_chunks;
      J.w_off = L.w_off; J.ld = L.ld; J.nrows = L.n_halves * 128;
      J.cons_inc = 2 / readers[g];
      if (part == 0) {
        J.b_off = P.layer[g - 1].stash_off; J.b_chunks = L.n_act_chunks;
        J.col0 = 0; J.ncols = L.n_act_chunks * 64;
      } else {
        J.b_off = (L.epi == EPI_BRANCH) ? P.stash_aux_dir_off : P.stash_aux_pos_off;
        J.b_chunks = 1; J.col0 = L.n_act_chunks * 64; J.ncols = L.ld - J.col0;
      }
      // cycles a wgrad CTA spends per tile: its MMAs (M = 128 per a-chunk pair, N = 64 per
      // b-chunk: N/2 cycles per K = 16 step, 8 steps per tile) plus a per-tile overhead that the
      // stage ring does not hide (swept 0-12000 cycles: 1500 is ~15 % slower, 3000 and up are flat)
      cost[WP.n_jobs] = (J.a_chunks / 2) * 8 * (J.b_chunks * 32) + kJobOverheadCycles;
      total += cost[WP.n_jobs];
      ++WP.n_jobs;
    }
  }
  sp = split_roles(WP.n_jobs, n_tiles);
  // CTAs per job proportional to its per-tile cycles; every job must keep up with the dgrad CTAs
  // (a late reader stalls them through the ring), so the CTAs left over by rounding go, one at a
  // time, to the job with the most cycles per CTA
  int n_cta[kMaxJobs], used = 0;
  for (int jn = 0; jn < WP.n_jobs; ++jn) {
    int n = (int)(sp.n_w * cost[jn] / total);
    if (n < 1) n = 1;
    if (n > sp.n_d) n = sp.n_d;  // a wgrad CTA serves whole dgrad CTAs
    n_cta[jn] = n;
    used += n;
  }
  while (used > sp.n_w) {  // rounding up the small jobs overshot: take from the best-served job
    int best = -1;
    for (int jn = 0; jn < WP.n_jobs; ++jn)
      if (n_cta[jn] > 1 && (best < 0 || cost[jn] / n_cta[jn] < cost[best] / n_cta[best])) best = jn;
    if (best < 0) break;
    --n_cta[best];
    --used;
  }
  while (used < sp.n_w) {
    int best = -1;
    for (int jn = 0; jn < WP.n_jobs; ++jn)
      if (n_cta[jn] < sp.n_d && (best < 0 || cost[jn] / n_cta[jn] > cost[best] / n_cta[best])) best = jn;
    if (best < 0) break;
    ++n_cta[best];
    ++used;
  }
  int begin = 0;
  for (int jn = 0; jn < WP.n_jobs; ++jn) {
    WP.job[jn].cta_begin = begin;
    WP.job[jn].n_split = n_cta[jn];
    begin += n_cta[jn];
  }
  WP.n_ctas = begin;
  return FSNERF_OK;
}

// bytes of the default workspace: flags, tile table, dpre ring
int64_t ring_workspace_bytes(const MlpProgram& P, const SplitB& sp, int64_t n_tiles) {
  return (int64_t)kFlagBytes + tile_table_bytes(n_tiles, sp.n_d) +
         (int64_t)sp.n_d * ring_depth_for(P.n_gemm) * kImgSlotBytes;
}

// Deterministic mode: the partial sums follow the default workspace (offsets in floats from
// there, each region 1 KB aligned): dW of every wgrad CTA, the dgrad CTAs' bias sums
// [n_d][4][n_gemm][256], the heads blocks' sums [hgrid][kHeadPart].
struct DetLayout {
  int64_t wpart_off[kMaxJobs];
  int64_t bpart_off, hpart_off, n_floats;
};
DetLayout det_layout(const MlpProgram& P, const WgradPlan& WP, const SplitB& sp, int64_t n_tiles) {
  DetLayout D;
  auto align = [](int64_t f) { return (f + 255) & ~(int64_t)255; };
  int64_t f = 0;
  for (int jn = 0; jn < WP.n_jobs; ++jn) {
    D.wpart_off[jn] = f;
    f += (int64_t)WP.job[jn].n_split * WP.job[jn].nrows * WP.job[jn].ncols;
  }
  for (int jn = WP.n_jobs; jn < kMaxJobs; ++jn) D.wpart_off[jn] = f;
  D.bpart_off = f = align(f);
  f += (int64_t)sp.n_d * 4 * P.n_gemm * 256;
  D.hpart_off = f = align(f);
  f += (int64_t)heads_grid(n_tiles) * kHeadPart;
  D.n_floats = align(f);
  return D;
}

}  // namespace
}  // namespace fs

using namespace fs;

extern "C" int64_t fsnerf_mlp_bwd_workspace_bytes(const fsnerf_net_cfg* cfg, int64_t n_samples) {
  MlpProgram P;
  if (build_program(cfg, &P) != FSNERF_OK) return -1;
  if (n_samples <= 0) return kFlagBytes;
  const int64_t n_tiles = (n_samples + kTileM - 1) / kTileM;
  const SplitB sp = split_roles(count_jobs(P), n_tiles);
  return (int64_t)kFlagBytes + tile_table_bytes(n_tiles, sp.n_d) +
         (int64_t)sp.n_d * ring_depth_for(P.n_gemm) * kImgSlotBytes;
}

extern "C" int64_t fsnerf_mlp_bwd_workspace_bytes_deterministic(const fsnerf_net_cfg* cfg, int64_t n_samples) {
  MlpProgram P;
  if (build_program(cfg, &P) != FSNERF_OK) return -1;
  if (n_samples <= 0) return kFlagBytes;
  const int64_t n_tiles = (n_samples + kTileM - 1) / kTileM;
  WgradPlan WP;
  SplitB sp;
  if (build_wgrad_plan(P, n_tiles, WP, sp) != FSNERF_OK) return -1;
  return ring_workspace_bytes(P, sp, n_tiles) + 4 * det_layout(P, WP, sp, n_tiles).n_floats;
}

namespace {
template <bool kDet>
int mlp_backward_impl(const fsnerf_net_cfg* cfg, const float* params, const void* packed, int64_t n_samples,
                      const void* stash, const float* out, const float* d_out, int density_only, float* grads,
                      void* workspace, void* stream) {
  MlpProgram P;
  int rc = build_program(cfg, &P);
  if (rc != FSNERF_OK) return rc;
  if (density_only) {
    fsnerf_set_error("mlp_backward: density_only backward is not supported (the reference's sigma_fn "
                     "pass runs under no_grad, src/render/rendering.py:58-64)");
    return FSNERF_ERR_UNSUPPORTED;
  }
  FS_REQUIRE(n_samples >= 0, "mlp_backward: negative n_samples");
  if (n_samples == 0) return FSNERF_OK;
  FS_REQUIRE(params && packed && stash && out && d_out && grads && workspace,
             "mlp_backward: null pointer");
  FS_REQUIRE(((reinterpret_cast<uintptr_t>(stash) | reinterpret_cast<uintptr_t>(workspace) |
               reinterpret_cast<uintptr_t>(packed)) & 127) == 0 &&
                 ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(d_out) |
                   reinterpret_cast<uintptr_t>(params)) & 15) == 0,
             "mlp_backward: stash/workspace/packed must be 128B aligned, out/d_out/params 16B");
  FS_REQUIRE(P.n_gemm <= kMaxLayersB, "mlp_backward: at most %d GEMM layers are supported", kMaxLayersB);
  cudaStream_t st = (cudaStream_t)stream;
  {  // function attributes are per device
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
      cudaError_t e = cudaFuncSetAttribute(mlp_bwd_fused_kernel<kDet>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           kSmemFused);
      if (e != cudaSuccess) {
        fsnerf_set_error("mlp_backward: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return FSNERF_ERR_CUDA;
      }
      if (dev >= 0 && dev < 64) configured[dev] = true;
    }
  }
  const int64_t n_tiles = (n_samples + kTileM - 1) / kTileM;

  // ---- wgrad plan and, in deterministic mode, where the partial sums go
  WgradPlan WP;
  SplitB sp;
  rc = build_wgrad_plan(P, n_tiles, WP, sp);
  if (rc != FSNERF_OK) return rc;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  float* parts = reinterpret_cast<float*>(ws + ring_workspace_bytes(P, sp, n_tiles));
  DetLayout DL;
  DetB det;
  det.wpart = det.bpart = nullptr;
  det.n_gemm = P.n_gemm;
  for (int jn = 0; jn < kMaxJobs; ++jn) det.wpart_off[jn] = 0;
  if constexpr (kDet) {
    DL = det_layout(P, WP, sp, n_tiles);
    det.wpart = parts;
    for (int jn = 0; jn < kMaxJobs; ++jn) det.wpart_off[jn] = DL.wpart_off[jn];
    det.bpart = parts + DL.bpart_off;
  }

  // ---- heads (sigma / rgb head weight gradients)
  HeadsArgs ha;
  ha.stash = reinterpret_cast<const uint8_t*>(stash); ha.stash_tile_bytes = P.stash_tile_bytes;
  ha.h_off = P.layer[P.n_hidden - 1].stash_off; ha.hb_off = P.layer[P.n_gemm - 1].stash_off;
  ha.n_samples = n_samples; ha.n_tiles = n_tiles; ha.out = out; ha.d_out = d_out;
  ha.g_sigma_w = grads + P.sigma_w_off; ha.g_sigma_b = grads + P.sigma_b_off;
  ha.g_rgb_w = grads + P.rgb_w_off; ha.g_rgb_b = grads + P.rgb_b_off;
  const int hgrid = heads_grid(n_tiles);
  {
    FsProfScope prof_("mlp_heads_wgrad", stream);
    float* hpart = nullptr;
    if constexpr (kDet) hpart = parts + DL.hpart_off;
    mlp_heads_wgrad_kernel<kDet><<<hgrid, 256, 0, st>>>(ha, hpart);
  }
  rc = fsnerf_check_launch("mlp_backward(heads)");
  if (rc != FSNERF_OK) return rc;

  // ---- dgrad plan + issue table
  PlanB PL;
  IssueTable T;
  PL.n_steps = P.n_gemm - 1;
  PL.g_branch = P.n_gemm - 1;
  PL.branch_mask_off = P.layer[P.n_gemm - 1].mask_off;
  int j = 0;
  int n_cons[4] = {0, 0, 0, 0};
  for (int s = 0; s < PL.n_steps; ++s)
    for (int c = 0; c < P.layer[P.n_gemm - 1 - s].bwd_n_chunks; ++c) ++n_cons[c];
  int cons[4] = {0, 0, 0, 0};
  for (int s = 0; s < PL.n_steps; ++s) {
    const int src = P.n_gemm - 1 - s, tgt = src - 1;
    StepB& S = PL.step[s];
    S.target = tgt;
    S.mask_off = P.layer[tgt].mask_off;
    S.add_sigma = (P.layer[tgt].epi == EPI_RELU_SIGMA) ? 1 : 0;
    const int nch = P.layer[src].bwd_n_chunks;
    FS_REQUIRE(P.layer[src].bwd_n_halves == 2 && nch <= 4 && j + nch <= kMaxChunks2,
               "mlp_backward: unsupported layer shape for the tensor-memory dgrad");
    for (int c = 0; c < nch; ++c, ++j) {
      IssueRec& R = T.rec[j];
      // a_ready[c] completes once per producer of chunk c (seed or a step's epilogue) and is
      // consumed once per step with more than c chunks: index = tile_iter * n_cons[c] + cons[c]
      R.flags = ((uint32_t)s << 24) | ((s & 1) ? kRecDcol : 0u) | (c == 0 ? kRecFirst : 0u) |
                (c == nch - 1 ? kRecLast : 0u) | kRecTmem | ((uint32_t)(cons[c] & 1) << kRecParShift) |
                ((n_cons[c] & 1) ? kRecParTile : 0u);
      R.idesc = umma_idesc_bf16(128, 256, 0, 0);
      R.a0 = (uint32_t)((s + 1) & 1) * 256u + 64u * c;
      R.abar = BarsB::a_ready + 8 * c;
      R.xbar = 0;
      R.accbar = BarsB::acc_full + 8 * (s & 1);
      R.n_acc = issue_n_acc(c, nch);
      R.w_block = (uint32_t)(P.layer[src].bwd_first_block + c * 2);
      R.w_bytes = kStageBytes;
      R.pad[0] = R.pad[1] = R.pad[2] = 0;
      ++cons[c];
    }
  }
  T.n = j;
  T.last_acc_off = BarsB::acc_full + 8 * ((PL.n_steps - 1) & 1);
  T.last_acc_n = 0;
  T.pad = 0;
  for (int s = 0; s < PL.n_steps; ++s)
    if ((s & 1) == ((PL.n_steps - 1) & 1)) ++T.last_acc_n;

  // ---- ring + flags in the caller's workspace
  RingB RG;
  RG.n_d = sp.n_d;
  RG.depth = ring_depth_for(P.n_gemm);
  RG.n_img = P.n_gemm;
  RG.prod = reinterpret_cast<uint32_t*>(ws);
  RG.tile_ctr = RG.prod + 255;
  RG.cons = RG.prod + 256;
  RG.row_cap = tile_row_cap(n_tiles, sp.n_d);
  RG.tile_of = reinterpret_cast<int32_t*>(ws + kFlagBytes);
  RG.base = ws + kFlagBytes + tile_table_bytes(n_tiles, sp.n_d);
  static_assert((256 + kNumSMs * kMaxRingDepth) * 4 <= kFlagBytes, "flag block too small");
  {
    cudaError_t e = cudaMemsetAsync(ws, 0, kFlagBytes, st);
    if (e != cudaSuccess) {
      fsnerf_set_error("mlp_backward: flag reset: %s", cudaGetErrorString(e));
      return FSNERF_ERR_CUDA;
    }
  }
  ArgsB a;
  a.trace = reinterpret_cast<long long*>(fsnerf_debug_trace_ptr());
  a.packed = reinterpret_cast<const uint8_t*>(packed);
  a.n_samples = n_samples;
  a.stash = reinterpret_cast<const uint8_t*>(stash);
  a.out = out; a.d_out = d_out; a.grads = grads;

  // every CTA of the launch must be resident at once (the roles wait on each other): one CTA
  // per SM, at most 148 of them, launched cooperatively so that the driver refuses instead of
  // deadlocking if that ever does not hold
  const int grid = sp.n_d + WP.n_ctas;
  void* kargs[] = {(void*)&P, (void*)&PL, (void*)&a, (void*)&T, (void*)&WP, (void*)&RG, (void*)&det};
  {
    FsProfScope prof_("mlp_bwd_fused", stream);
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)mlp_bwd_fused_kernel<kDet>, dim3(grid), dim3(kThreadsB),
                                                kargs, (size_t)kSmemFused, st);
    if (e != cudaSuccess) {
      fsnerf_set_error("mlp_backward: cooperative launch of %d CTAs failed: %s", grid, cudaGetErrorString(e));
      return FSNERF_ERR_CUDA;
    }
  }
  rc = fsnerf_check_launch("mlp_backward(fused)");
  if (rc != FSNERF_OK || !kDet) return rc;

  // ---- deterministic mode: every element's partials, in index order, added to grads once
  RedPlan RP;
  RP.n = 0;
  int64_t most = 0;
  auto seg = [&](int64_t dst, int64_t src, int64_t part_stride, int rows, int cols, int dst_ld, int src_ld,
                 int n_parts) {
    RedSeg& S = RP.seg[RP.n++];
    S.dst = dst; S.src = src; S.part_stride = part_stride;
    S.rows = rows; S.cols = cols; S.dst_ld = dst_ld; S.src_ld = src_ld; S.n_parts = n_parts;
    if ((int64_t)rows * cols > most) most = (int64_t)rows * cols;
  };
  for (int jn = 0; jn < WP.n_jobs; ++jn) {  // weights: the job's wgrad CTAs in CTA order
    const WgradJob& J = WP.job[jn];
    seg(J.w_off + J.col0, DL.wpart_off[jn], (int64_t)J.nrows * J.ncols, J.nrows, J.ncols, J.ld, J.ncols, J.n_split);
  }
  for (int g = 0; g < P.n_gemm; ++g)  // biases: the dgrad CTAs in CTA order
    seg(P.layer[g].bias_off, DL.bpart_off + g * 256, (int64_t)4 * P.n_gemm * 256, 1, P.layer[g].n_halves * 128, 0, 0,
        sp.n_d);
  // heads: the blocks in block order
  seg(P.sigma_w_off, DL.hpart_off, kHeadPart, 1, 256, 0, 0, hgrid);
  seg(P.rgb_w_off, DL.hpart_off + 256, kHeadPart, 1, 384, 0, 0, hgrid);
  seg(P.rgb_b_off, DL.hpart_off + 640, kHeadPart, 1, 3, 0, 0, hgrid);
  seg(P.sigma_b_off, DL.hpart_off + 643, kHeadPart, 1, 1, 0, 0, hgrid);
  {
    FsProfScope prof_("mlp_bwd_det_reduce", stream);
    const int gx = (int)((most + 255) / 256 < 256 ? (most + 255) / 256 : 256);
    mlp_bwd_det_reduce_kernel<<<dim3(gx, RP.n), 256, 0, st>>>(RP, parts, grads);
  }
  return fsnerf_check_launch("mlp_backward(deterministic reduction)");
}
}  // namespace

extern "C" int fsnerf_mlp_backward(const fsnerf_net_cfg* cfg, const float* params,
                                   const void* packed, int64_t n_samples, const void* stash,
                                   const float* out, const float* d_out, int density_only,
                                   float* grads, void* workspace, void* stream) {
  return mlp_backward_impl<false>(cfg, params, packed, n_samples, stash, out, d_out, density_only, grads, workspace,
                                  stream);
}

extern "C" int fsnerf_mlp_backward_deterministic(const fsnerf_net_cfg* cfg, const float* params,
                                                 const void* packed, int64_t n_samples, const void* stash,
                                                 const float* out, const float* d_out, int density_only,
                                                 float* grads, void* workspace, void* stream) {
  return mlp_backward_impl<true>(cfg, params, packed, n_samples, stash, out, d_out, density_only, grads, workspace,
                                 stream);
}
