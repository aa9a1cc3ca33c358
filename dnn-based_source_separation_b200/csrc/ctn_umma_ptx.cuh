// Raw PTX wrappers for the Blackwell (sm_100a) features the pointwise kernels use: mbarrier, 1-D bulk async copy
// (TMA engine, UBLKCP), tcgen05 alloc / mma / commit / ld, proxy fences.  No CUTLASS dependency.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}

// ---- async proxy -----------------------------------------------------------------------------------------------
// generic-proxy st.shared writes -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 1-D bulk copy global -> shared, completion on an mbarrier (complete_tx::bytes).  size % 16 == 0, 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// one lane of a converged warp (elect.sync): code under this predicate is known single-threaded to the compiler, so
// uniform-datapath instructions (tcgen05.mma / commit) are emitted without per-instruction election loops
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 rx;\n\t"
      ".reg .pred px;\n\t"
      "elect.sync rx|px, 0xFFFFFFFF;\n\t"
      "@px mov.s32 %0, 1;\n\t"
      "}"
      : "+r"(pred));
  return pred != 0;
}

// ---- clusters ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of every CTA in the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// wait with acquire at CLUSTER scope (the arrivals may come from the peer CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}

// bulk copy from this CTA's shared memory into the SAME offsets of CTA `rank` of the cluster (distributed shared memory), completing
// on the mbarrier at `bar` (CTA-relative address) in that CTA: the transfer runs in the async proxy on both sides, so the
// receiver's tcgen05.mma may read the data right after its mbarrier wait.  16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_s2peer(uint32_t dst_smem, uint32_t src_smem, uint32_t bytes, uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t"
      ".reg .b32 rd, rb;\n\t"
      "mapa.shared::cluster.u32 rd, %0, %4;\n\t"
      "mapa.shared::cluster.u32 rb, %3, %4;\n\t"
      "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [rd], [%1], %2, [rb];\n\t"
      "}" ::"r"(dst_smem), "r"(src_smem), "r"(bytes), "r"(bar), "r"(rank)
      : "memory");
}

// ---- tcgen05 ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp (the allocating one)
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, kind::tf32, issued by ONE thread
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with fp16 operands (K = 16 per instruction, twice the rate of kind::tf32)
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// same, arriving on the barrier at this CTA-relative offset in every CTA of cta_mask
__device__ __forceinline__ void mma_commit_multicast(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(cta_mask)
               : "memory");
}

// 32 lanes x 32 columns of fp32: thread i of the warp receives columns [col, col+32) of TMEM lane (base_lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
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
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- A operand in tensor memory ("ts" form) ------------------------------------------------------------------------
// D[tmem] (+)= A[tmem] * B[smem desc]^T, kind::f16.  A: lane = row m, 32-bit column j = {A[m][2j] (low half), A[m][2j+1]}; one
// instruction consumes 8 columns (K = 16).  Layout verified on B200 with tools/umma_unit_ts.cu.
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// thread i of the warp writes 8 consecutive 32-bit columns of TMEM lane (base_lane + i)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// round-to-nearest fp32 -> tf32 (result is an fp32 bit pattern with the low 13 mantissa bits cleared)
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// fp16 hi/lo split of two fp32 values ("3xFP16"): hi = rn_f16(x) (saturating, never inf), lo = rn_f16(x - hi).
// Both pieces carry 11 significant bits like TF32; packed as f16x2 (element 0 in the low half).
__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
  float h0, h1;
  asm("{\n\t.reg .f16 a, b;\n\tmov.b32 {a, b}, %2;\n\tcvt.f32.f16 %0, a;\n\tcvt.f32.f16 %1, b;\n\t}" : "=f"(h0), "=f"(h1) : "r"(hi));
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - h1), "f"(x0 - h0));
}

// cheap hi piece for the 3xTF32 scheme (3 instructions per element instead of an emulated cvt.rna): x rounded to nearest
// (ties away) at 10 explicit mantissa bits via integer add + mask; lo = x - hi is EXACT in fp32 and the tensor core consumes
// its leading tf32 bits (remaining error <= 2^-21 |x|).
__device__ __forceinline__ float hi_tf32(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }

// ---- descriptors -------------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor (sm_100 "version 1"), SWIZZLE_128B canonical layouts:
//   bits [0,14) start address >> 4 | [16,30) leading byte offset >> 4 | [32,46) stride byte offset >> 4
//   [46,48) version = 1 | [49,52) base offset = 0 | [61,64) layout type (2 = SWIZZLE_128B)
//   layout types: 2 = SWIZZLE_128B (16-byte chunks XOR row%8; K-major tf32 and all 16-bit operands),
//                 1 = SWIZZLE_128B_BASE32B (32-byte chunks XOR row%4) -- the ONLY layout the hardware accepts for
//                     MN-major 32-bit (tf32) operands (measured: SWIZZLE_128B MN-major tf32 returns zeros).
__host__ __device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                            uint32_t layout_type = 2) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout_type << 61;
  return d;
}
// Instruction descriptor for kind::tf32, fp32 accumulate, M = 128:
//   [4,6) c_format = 1 (F32) | [7,10) a_format = 2 (TF32) | [10,13) b_format = 2 | [15] a_major | [16] b_major
//   [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// kind::f16 with F16 inputs (a_format = b_format = 0), fp32 accumulate
__host__ __device__ __forceinline__ uint32_t make_idesc_f16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

}  // namespace ptx
