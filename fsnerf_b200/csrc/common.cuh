// Shared device helpers for the fsnerf_b200 kernels (sm_100a only).
// PTX wrappers for mbarrier, bulk async copy (TMA engine), tcgen05 / TMEM.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#define FSNERF_OK 0
#define FSNERF_ERR_ARG -1
#define FSNERF_ERR_CUDA -2
#define FSNERF_ERR_UNSUPPORTED -3

void fsnerf_set_error(const char* fmt, ...);
void* fsnerf_debug_trace_ptr();
int fsnerf_check_launch(const char* what);

#define FS_REQUIRE(cond, ...)                 \
  do {                                        \
    if (!(cond)) {                            \
      fsnerf_set_error(__VA_ARGS__);          \
      return FSNERF_ERR_ARG;                  \
    }                                         \
  } while (0)

// Optional per-kernel device timing (cudaEvents on the launch stream), enabled by
// fsnerf_profile_enable(); bench.py uses it for the live roofline numbers.
struct FsProfScope {
  FsProfScope(const char* name, void* stream);
  ~FsProfScope();
  int slot;
  void* stream;
};

namespace fs {

constexpr int kNumSMs = 148;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
// No suspend-time hint: with one, ptxas emits TRYWAIT + NANOSLEEP.SYNCS and the wake-up
// latency of the sleeping warp lands on the critical path of every hand-over (measured: -12 %
// on the fused MLP forward).
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded spin: a protocol bug turns into a trap (reported as a launch error)
// instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) {
      printf("fsnerf: mbarrier timeout blk %d thr %d bar %u parity %u\n", blockIdx.x, threadIdx.x,
             bar, parity);
      __trap();
    }
  }
}

// For warps that are NOT on the critical path (weight producers, store warps, encoders): back
// off between polls so that the spin loop does not take issue slots from the epilogue and
// MMA-issuer warps sharing the scheduler.
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(128);
    if (++spins > (1u << 22)) {
      printf("fsnerf: mbarrier timeout blk %d thr %d bar %u parity %u\n", blockIdx.x, threadIdx.x,
             bar, parity);
      __trap();
    }
  }
}

// Same, for a warp that must stay provably CONVERGED (the MMA issuer): the loop exit is a
// warp vote, so the compiler's divergence analysis keeps everything downstream uniform
// (operands of the tcgen05 instructions then live in uniform registers).
__device__ __forceinline__ void mbar_wait_converged(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!__all_sync(0xffffffffu, mbar_try_wait(bar, parity))) {
    if (++spins > (1u << 24)) {
      if ((threadIdx.x & 31) == 0)
        printf("fsnerf: mbarrier timeout blk %d thr %d bar %u parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- register re-split per role
// (warpgroup granularity: all four warps of an aligned group must execute the same one)
template <int kRegs> __device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs));
}
template <int kRegs> __device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs));
}

// ---------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------- bulk async copy (TMA engine, SASS UBLKCP)
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes,
                                         uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(dst_smem),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
               "r"(src_smem), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read0() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait0() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------- TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets TMEM lane
// (taddr.lane + i), columns taddr.col .. +31.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// ---------------------------------------------------------------- UMMA (tcgen05.mma)
// Shared-memory matrix descriptor, SWIZZLE_128B canonical layouts
// (cute/arch/mma_sm100_desc.hpp SmemDescriptor): start>>4 [0,14), LBO>>4
// [16,30), SBO>>4 [32,46), version=1 [46,48), layout_type=2 (SW128) [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                    uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor for kind::f16, bf16 x bf16 -> f32 (InstrDescriptor).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major,
                                                       int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) |
         ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand read from TMEM (lane = row, one 32-bit column = two consecutive bf16 K
// elements; K=16 per instruction = 8 columns), B from a shared-memory descriptor.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// One lane of a converged warp, chosen by the hardware: inside `if (elect_one())` the compiler knows
// a single thread is active, so register operands move to the uniform datapath with plain R2UR
// (no ELECT + R2UR.BROADCAST loop per tcgen05 instruction).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// Converged-issue forms: executed by ALL lanes of the issuing warp with a per-lane guard that is
// true for one lane only.  In the micro-benchmark (tools/mma_bench.cu) the operands stayed in
// uniform registers (128.0 cycles per M=128 N=256 K=16 MMA vs 138 from a lane-0 branch); in the
// real kernels the compiler still wrapped each one in an ELECT + R2UR.BROADCAST loop, so the MLP
// kernels issue from `if (elect_one())` instead (above).  Kept for the benchmarks.
__device__ __forceinline__ void umma_bf16_ts_conv(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b,
                                                  uint32_t idesc, uint32_t accumulate, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(issue)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_conv(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                                  uint32_t idesc, uint32_t accumulate, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 e, %5, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(issue)
      : "memory");
}
// Two MMAs with two NON-BLOCKING mbarrier probes slotted between them (converged issue).
// The tensor pipe accepts the next MMA only when the previous one is (nearly) done and has
// < 100 cycles of slack before it idles (tools/mma_bench.cu), so everything the issuing warp
// must do for the NEXT chunk (iterator advance, descriptors, readiness tests) is placed
// between the MMA issues of the current chunk, never between chunks.
template <bool kATmem>
__device__ __forceinline__ void umma2_probe(uint32_t tmem_d, uint64_t a0, uint64_t a1, uint64_t b0, uint64_t b1,
                                            uint32_t idesc, uint32_t issue, uint32_t bar0, uint32_t par0,
                                            uint32_t bar1, uint32_t par1, uint32_t& ok0, uint32_t& ok1) {
  if (kATmem) {
    asm volatile(
        "{\n\t.reg .pred e, t, q0, q1;\n\t"
        "setp.ne.b32 e, %8, 0;\n\t"
        "setp.eq.b32 t, %8, %8;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%2], [%3], %5, %7, t;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 q0, [%9], %10;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 q1, [%11], %12;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%2], [%4], %6, %7, t;\n\t"
        "selp.u32 %0, 1, 0, q0;\n\t"
        "selp.u32 %1, 1, 0, q1;\n\t}"
        : "=r"(ok0), "=r"(ok1)
        : "r"(tmem_d), "r"((uint32_t)a0), "r"((uint32_t)a1), "l"(b0), "l"(b1), "r"(idesc), "r"(issue),
          "r"(bar0), "r"(par0), "r"(bar1), "r"(par1)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred e, t, q0, q1;\n\t"
        "setp.ne.b32 e, %8, 0;\n\t"
        "setp.eq.b32 t, %8, %8;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%2], %3, %5, %7, t;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 q0, [%9], %10;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 q1, [%11], %12;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%2], %4, %6, %7, t;\n\t"
        "selp.u32 %0, 1, 0, q0;\n\t"
        "selp.u32 %1, 1, 0, q1;\n\t}"
        : "=r"(ok0), "=r"(ok1)
        : "r"(tmem_d), "l"(a0), "l"(a1), "l"(b0), "l"(b1), "r"(idesc), "r"(issue),
          "r"(bar0), "r"(par0), "r"(bar1), "r"(par1)
        : "memory");
  }
}
// low word of a SWIZZLE_128B K-major descriptor (start address, LBO = 16 B) and the
// constant high word (SBO = 1024 B, version 1, layout SW128): desc = hi:lo, and advancing
// by 32 bytes along K adds 2 to the low word
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_addr) {
  return ((smem_addr >> 4) & 0x3FFFu) | (1u << 16);
}
constexpr uint32_t kUmmaDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t umma_desc_from_lo(uint32_t lo) {
  return ((uint64_t)kUmmaDescHiSw128 << 32) | lo;
}
__device__ __forceinline__ void umma_commit_conv(uint32_t bar, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "setp.ne.b32 e, %1, 0;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar),
      "r"(issue)
      : "memory");
}
// registers -> TMEM: thread i of the warp writes lane (taddr.lane + i), 16 consecutive columns
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
      "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read1() {
  asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   bar)
               : "memory");
}

// ---------------------------------------------------------------- SW128 tile addressing
// A [rows x 64 bf16] K-major SWIZZLE_128B tile: row r is 128 B; 16-byte unit j
// of the row lives at unit (j ^ (r & 7)).  Tiles are 1024 B aligned.
__host__ __device__ __forceinline__ uint32_t sw128_off(uint32_t row, uint32_t unit16) {
  return row * 128u + ((unit16 ^ (row & 7u)) << 4);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// relu fused into the fp32 -> bf16x2 conversion
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// packed fp32 add (sm_100: one FADD2 for two lanes)
__device__ __forceinline__ void add_f32x2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
  asm("{\n\t.reg .b64 ra, rb, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\t"
      "mov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d0), "=f"(d1)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c),
               "r"(d)
               : "memory");
}

}  // namespace fs
