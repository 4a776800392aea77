// umma.cuh - thin inline-PTX wrappers for the sm_100a tensor path: mbarrier, tcgen05 (alloc / mma
// kind::i8 / commit / ld), proxy fences, shared-memory matrix descriptors.
// Written for sm_100a only (no other arch is ever compiled).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace pl2 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------- mbarrier ----------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  // make barrier initialisation visible to the async proxy (tcgen05.commit arrives through it)
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
// One arrival per WARP (barrier count = producer warps): mbarrier.arrive is a shared-memory atomic,
// and one per thread (288 per k-step in the first TS kernel) serialises on the barrier word.  Each
// lane orders its own writes first (fence.proxy.async / tcgen05.wait::st + fence), __syncwarp makes
// them cumulative with lane 0's release-arrive.
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar, uint32_t lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
}
// NOTE on releasing a shared-memory ring slot the lanes have READ with ld.shared: arrive only after an instruction
// that consumed the loaded registers has issued (st.shared / tcgen05.st of values derived from them).  An arrive
// placed right after the loads can overtake them in the memory pipeline.
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---------------- TMA (bulk async copies completing on an mbarrier) ----------------
// expect_tx: one arrival + the number of bytes the bulk copies issued next will deliver.
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 2-D tiled tensor-map load (SASS UTMALDG): box at element coordinates {c0 (innermost), c1} -> dense
// shared-memory box, completes `box bytes` on the mbarrier.
__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const void* tensor_map, int32_t c0, int32_t c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst_smem), "l"(tensor_map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst_smem, const void* tensor_map, int32_t c0, int32_t c1, int32_t c2, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst_smem), "l"(tensor_map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)) : "memory");
}
// 1-D bulk copy global -> shared (SASS UBLKCP); bytes and both addresses multiples of 16.
__device__ __forceinline__ void bulk_load_1d(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// Asynchronous bulk reduction shared -> global through the TMA unit (SASS UBLKRED): global[i] += smem[i] on
// 32-bit signed integers / fp64, performed at the L2 without the SM ever reading the old values.  Issued by one
// thread; completion of the shared-memory READS is tracked by that thread's bulk async-groups.
__device__ __forceinline__ void bulk_reduce_add_s32(void* dst_global, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.s32 [%0], [%1], %2;" ::"l"(dst_global), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_reduce_add_f64(void* dst_global, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], %2;" ::"l"(dst_global), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
// named barrier among a subset of the CTA's warps (id 1..15; thread count a multiple of 32)
template <uint32_t kId, uint32_t kThreads>
__device__ __forceinline__ void named_bar_sync() {
  asm volatile("bar.sync %0, %1;" ::"n"(kId), "n"(kThreads) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t addr, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory"); }
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void prefetch_tensormap(const void* tensor_map) { asm volatile("prefetch.tensormap [%0];" ::"l"(tensor_map) : "memory"); }
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts64x2(uint32_t addr, uint32_t lo, uint32_t hi) { asm volatile("st.shared.v2.b32 [%0], {%1,%2};" ::"r"(addr), "r"(lo), "r"(hi) : "memory"); }
// F32 accumulator bits -> int32, round to nearest (exact for the integer values below 2^24 the FP4 kernels produce)
__device__ __forceinline__ int32_t f32_bits_to_s32_rn(uint32_t bits) {
  int32_t r;
  asm("cvt.rni.s32.f32 %0, %1;" : "=r"(r) : "f"(__uint_as_float(bits)));
  return r;
}

// ---------------- fences ----------------
// generic-proxy st.shared -> visible to the async proxy (UMMA operand fetch)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---------------- TMEM allocation (one full warp executes these) ----------------
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {
  static_assert(kCols == 32 || kCols == 64 || kCols == 128 || kCols == 256 || kCols == 512, "TMEM columns: power of two >= 32");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(kCols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// ---------------- descriptors ----------------
// Shared-memory matrix descriptor, SWIZZLE_NONE ("interleave") canonical layout.  Field layout
// per the PTX ISA tcgen05 matrix-descriptor table (also cute/arch/mma_sm100_desc.hpp:103-130):
//   [0,14)  start address >> 4        [16,30) leading-dimension byte offset >> 4
//   [32,46) stride-dimension byte offset >> 4   [46,48) version = 1 on sm_100
//   [49,52) base offset = 0           [61,64) layout type (0 = no swizzle)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}

// Instruction descriptor for kind::i8 (cute/arch/mma_sm100_desc.hpp:409-436 documents the bits):
//   [4,6) D format: 2 = S32   [7,10) A format: 1 = signed 8-bit   [10,13) B format
//   [15] A major: 1 = MN-major   [16] B major   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_i8(uint32_t m, uint32_t n, bool a_mn_major, bool b_mn_major, bool a_signed = true, bool b_signed = true) {
  return (2u << 4) | ((a_signed ? 1u : 0u) << 7) | ((b_signed ? 1u : 0u) << 10) | ((a_mn_major ? 1u : 0u) << 15) |
         ((b_mn_major ? 1u : 0u) << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_i8_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (count 1) on an mbarrier once all previously issued tcgen05.mma of this thread retire.
// Implies tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---------------- TMEM -> registers ----------------
// 32 lanes x 32-bit, 16 consecutive columns: thread t of the warp receives row (lane base + t).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace pl2

namespace pl2 {

// D[tmem] (+)= A[tmem] * B[smem]  ("TS" form: the A operand is read from tensor memory, K-major,
// lane = row, each 32-bit column = 4 consecutive K bytes); issued by ONE thread.
__device__ __forceinline__ void umma_i8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Instruction descriptor for kind::mxf4 (block-scaled E2M1, PTX ISA tcgen05 "instruction descriptor" table for
// the .kind::mxf8f6f4 / .kind::mxf4 forms):
//   [4,6) SF id of B (byte of the scale column)   [7,10) A format: 1 = E2M1   [10,12) B format: 1 = E2M1
//   [15] / [16] A / B major: 0 = K-major (the only layout 4-bit operands accept)
//   [17,23) N >> 3   [23] scale format: 1 = UE8M0   [24,29) M >> 4   [29,31) SF id of A   [31] K = 64
// D is always F32.  Callers that fill every scale byte with the same value can leave both SF ids at 0.
__host__ __device__ constexpr uint32_t make_idesc_mxf4(uint32_t m, uint32_t n) {
  return (1u << 7) | (1u << 10) | ((n >> 3) << 17) | (1u << 23) | ((m >> 4) << 24);
}

// D[tmem] (+)= (A[tmem] x 2^sfa) * (B[smem] x 2^sfb), K = 64 packed E2M1 per row (32 bytes = 8 TMEM columns of A),
// one UE8M0 scale per 32 K (scale_vec::2X) read from tensor memory at sfa / sfb; issued by ONE thread.
__device__ __forceinline__ void umma_mxf4_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t sfa_tmem, uint32_t sfb_tmem, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.scale_vec::2X [%0], [%1], %2, %3, [%4], [%5], p;\n\t}"
      :
      : "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(sfa_tmem), "r"(sfb_tmem), "r"(accumulate)
      : "memory");
}
// UE8M0 scale bytes of 2^0 (bias 127): with every scale byte set to this, a block-scaled product is the plain product
constexpr uint32_t kUe8m0One4 = 0x7F7F7F7Fu;

// registers -> TMEM: thread t of the warp writes 8 consecutive 32-bit columns of lane (lane base + t)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }


// ---- single-thread issue without waterfall loops -------------------------------------------------
// tcgen05.mma / tcgen05.commit are warp-level uniform-datapath instructions in SASS (UTCIMMA, UTCBAR).
// ptxas emits them straight-line only when (a) the surrounding control flow is provably warp-uniform
// and (b) every operand is provably uniform; otherwise EACH one is wrapped in a VOTEU / ELECT /
// R2UR.BROADCAST / BRA.U.ANY waterfall loop that costs 110-190 clk per UMMA on the issuing thread
// (umma_issue_bench_kernel: 186 clk/UMMA under `if (lane == 0)`, i.e. more than the 40-96 clk the
// tensor pipe needs for our N = 80..192 shapes).  Recipe, as in CUTLASS' sm100 kernels:
//   * take the warp index with uniform_warp_idx() (a __shfl_sync from lane 0 is provably uniform),
//   * broadcast values read from memory (the TMEM base) with uniform_u32(),
//   * run the issuer loop on the WHOLE warp and guard the tcgen05 block with `if (elect_one_sync())`.
__device__ __forceinline__ uint32_t uniform_u32(uint32_t v) { return __shfl_sync(0xFFFFFFFFu, v, 0); }
__device__ __forceinline__ uint32_t uniform_warp_idx() { return __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0); }
__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred = 0, laneid = 0;
  asm volatile(
      "{\n\t.reg .b32 %%rx;\n\t.reg .pred %%px;\n\t"
      "elect.sync %%rx|%%px, %2;\n\t"
      "@%%px mov.s32 %1, 1;\n\t"
      "mov.s32 %0, %%rx;\n\t}"
      : "+r"(laneid), "+r"(pred)
      : "r"(0xFFFFFFFFu));
  return pred;
}

}  // namespace pl2
