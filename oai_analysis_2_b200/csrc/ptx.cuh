// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (tiled + bulk), tcgen05 (alloc / mma / commit / ld).
// Only what the conv implicit-GEMM kernel needs; no CUTLASS dependency.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

namespace oai {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a lost arrive must become a trap with a message, never a hung GPU.
#ifndef OAI_MBAR_TIMEOUT_NS
#define OAI_MBAR_TIMEOUT_NS 4000000000ull
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag = 0) {
  if (mbar_try_wait(bar, parity)) return;
  // the clock is read only once per 2^16 failed polls, so the polling loop of the single-warp roles stays at a handful
  // of instructions (each try_wait already suspends the thread for a hardware-defined interval)
  uint64_t t0 = 0;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0xffff) == 0) {
      const uint64_t t = globaltimer_ns();
      if (t0 == 0) t0 = t;
      else if (t - t0 > OAI_MBAR_TIMEOUT_NS) {
        printf("[oai] mbarrier timeout: block %d thread %d tag %d parity %u\n", blockIdx.x, threadIdx.x, tag, parity);
        __trap();
      }
    }
  }
}

// 16-byte shared-memory load through the shared window (an LDS, not a generic LD): the compiler may schedule it freely
// against global stores
__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
      : "memory");
}
// 1-D bulk copy global -> shared (size multiple of 16, both 16-B aligned).
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T ; both operands K-major, kind::f16 (fp16 or bf16 inputs, fp32 accumulate).
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, with the two shared-memory descriptors given as (low word, shared high word): the high word (SBO, version,
// swizzle mode) is constant for a kernel and the low word (start address, LBO) is one integer add away from the
// stage base, which keeps the issue loop short.
__device__ __forceinline__ void umma_f16_ss_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi,
                                                 uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with a separate high word per operand (different SBO for A and B).
__device__ __forceinline__ void umma_f16_ss_lohi2(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                                  uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Block-scaled 8-bit form: D[tmem] (+)= (A * SFA) * (B * SFB)^T with A, B e4m3 (K = 32 per instruction, 32 bytes per
// row like a K = 16 fp16 step) and one UE8M0 scale per row and 32-wide K block read from TMEM at sfa / sfb.
__device__ __forceinline__ void umma_mxf8_ss_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi,
                                                  uint32_t idesc, uint32_t tmem_sfa, uint32_t tmem_sfb,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %7, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::mxf8f6f4.block_scale.scale_vec::1X [%0], da, db, %4, [%5], [%6], p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(tmem_sfa), "r"(tmem_sfb), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_mxf8_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t tmem_sfa, uint32_t tmem_sfb, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::mxf8f6f4.block_scale.scale_vec::1X [%0], %1, %2, %3, [%4], [%5], p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(tmem_sfa), "r"(tmem_sfb), "r"(accumulate)
      : "memory");
}
// mbarrier arrive once every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane (base_lane + t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 32 consecutive columns, every column of thread t's lane set to v
__device__ __forceinline__ void tmem_st_32x32_fill(uint32_t taddr, uint32_t v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
      "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
      :
      : "r"(taddr), "r"(v)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major, 128-byte swizzle (rows of 128 B, 8-row groups `sbo_bytes` apart).
// Field layout follows the sm_100 UMMA descriptor: [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4,
// [46,48) version=1, [49,52) base offset, [61,64) layout type (2 = SWIZZLE_128B).
// layout_type: 2 = SWIZZLE_128B (rows of 128 B, sbo 1024), 4 = SWIZZLE_64B (rows of 64 B, sbo 512).
__device__ __forceinline__ uint64_t umma_desc_kmajor(uint32_t smem_addr, uint32_t sbo_bytes, uint32_t base_offset,
                                                     uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;  // LBO (unused for swizzled K-major)
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(base_offset & 7) << 49;
  d |= static_cast<uint64_t>(layout_type & 7) << 61;
  return d;
}
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t sbo_bytes, uint32_t base_offset) {
  return umma_desc_kmajor(smem_addr, sbo_bytes, base_offset, 2);
}

// Instruction descriptor for kind::f16: fp32 accumulate, A/B both K-major.
// ab_format: 0 = fp16, 1 = bf16.
__device__ __host__ __forceinline__ uint32_t umma_idesc_f16(uint32_t M, uint32_t N, uint32_t ab_format) {
  uint32_t d = 0;
  d |= 1u << 4;                 // c_format = F32
  d |= (ab_format & 7u) << 7;   // a_format
  d |= (ab_format & 7u) << 10;  // b_format
  d |= (N >> 3) << 17;
  d |= (M >> 4) << 24;
  return d;
}

// Instruction descriptor for kind::mxf8f6f4 with block scaling: A and B e4m3 (format 0), K-major, fp32 accumulate,
// UE8M0 scale factors (bit 23), scale-factor byte 0 of A and B (bits [29,31) / [4,6)).
__device__ __host__ __forceinline__ uint32_t umma_idesc_mxf8_e4m3(uint32_t M, uint32_t N) {
  uint32_t d = 0;
  d |= (N >> 3) << 17;
  d |= 1u << 23;
  d |= (M >> 4) << 24;
  return d;
}

}  // namespace oai
