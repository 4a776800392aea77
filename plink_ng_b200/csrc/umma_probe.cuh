// umma_probe.cuh - single-CTA tcgen05 probe: runs int8 UMMAs over caller-supplied shared-memory
// images with caller-supplied descriptor fields and returns the TMEM accumulator.  Used by
// pl2gpu_selftest_umma (production layout vs scalar reference) and by tests/ to pin the operand
// layout the production kernels rely on.
#pragma once
#include "common.cuh"
#include "umma.cuh"

namespace pl2 {

struct UmmaProbeParams {
  uint32_t a_bytes, b_bytes;        // image sizes (A at smem offset 0, B at b_smem_off)
  uint32_t b_smem_off;              // multiple of 128
  uint32_t a_lbo, a_sbo, b_lbo, b_sbo;
  uint32_t a_step_bytes, b_step_bytes;  // descriptor start-address advance per k-step
  uint32_t k_steps;
  uint32_t idesc;
  uint32_t n;                       // columns to read back (multiple of 16, <= 256)
};

constexpr uint32_t kProbeSmemBytes = 96 * 1024;

__global__ void __launch_bounds__(128, 1)
umma_probe_kernel(const uint8_t* __restrict__ a_img, const uint8_t* __restrict__ b_img, UmmaProbeParams prm, int32_t* __restrict__ d_out /* [128][n] */) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done;
  __shared__ uint32_t tmem_base_slot;
  const uint32_t tid = threadIdx.x;
  const uint32_t warp = tid >> 5;
  const uint32_t lane = tid & 31;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  uint8_t* sm = smem + (smem_base - smem_u32(smem));
  for (uint32_t i = tid; i < prm.a_bytes; i += 128) sm[i] = a_img[i];
  for (uint32_t i = tid; i < prm.b_bytes; i += 128) sm[prm.b_smem_off + i] = b_img[i];
  if (tid == 0) {
    mbar_init(&bar_done, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<256>(&tmem_base_slot);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;
  if (tid == 0) {
    for (uint32_t ks = 0; ks < prm.k_steps; ++ks) {
      const uint64_t da = make_smem_desc(smem_base + ks * prm.a_step_bytes, prm.a_lbo, prm.a_sbo);
      const uint64_t db = make_smem_desc(smem_base + prm.b_smem_off + ks * prm.b_step_bytes, prm.b_lbo, prm.b_sbo);
      umma_i8_ss(tmem_base, da, db, prm.idesc, ks ? 1u : 0u);
    }
    umma_commit(&bar_done);
  }
  mbar_wait(&bar_done, 0);
  tc_fence_after_sync();
  for (uint32_t c0 = 0; c0 < prm.n; c0 += 16) {
    uint32_t v[16];
    tmem_ld16(tmem_base + ((32u * warp) << 16) + c0, v);
    tmem_ld_wait();
#pragma unroll
    for (uint32_t c = 0; c < 16; ++c) d_out[static_cast<uint64_t>(32 * warp + lane) * prm.n + c0 + c] = static_cast<int32_t>(v[c]);
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc<256>(tmem_base);
  }
}


// TS probe: A rows come from global memory ([128][k_steps*32] int8, K-major), are written to TMEM
// with tcgen05.st (8 columns per k-step at column 256 + 8*ks) and multiplied with the smem B image.
__global__ void __launch_bounds__(128, 1)
umma_probe_ts_kernel(const uint8_t* __restrict__ a_rows, const uint8_t* __restrict__ b_img, UmmaProbeParams prm, int32_t* __restrict__ d_out /* [128][n] */) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done;
  __shared__ uint32_t tmem_base_slot;
  const uint32_t tid = threadIdx.x;
  const uint32_t warp = tid >> 5;
  const uint32_t lane = tid & 31;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  uint8_t* sm = smem + (smem_base - smem_u32(smem));
  for (uint32_t i = tid; i < prm.b_bytes; i += 128) sm[i] = b_img[i];
  if (tid == 0) {
    mbar_init(&bar_done, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_base_slot);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;
  const uint32_t row_bytes = prm.k_steps * 32;
  for (uint32_t ks = 0; ks < prm.k_steps; ++ks) {
    uint32_t v[8];
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a_rows + static_cast<uint64_t>(tid) * row_bytes + ks * 32);
#pragma unroll
    for (uint32_t c = 0; c < 8; ++c) v[c] = src[c];
    tmem_st8(tmem_base + ((32u * warp) << 16) + 256 + 8 * ks, v);
  }
  tmem_st_wait();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (tid == 0) {
    for (uint32_t ks = 0; ks < prm.k_steps; ++ks) {
      const uint64_t db = make_smem_desc(smem_base + ks * prm.b_step_bytes, prm.b_lbo, prm.b_sbo);
      umma_i8_ts(tmem_base, tmem_base + 256 + 8 * ks, db, prm.idesc, ks ? 1u : 0u);
    }
    umma_commit(&bar_done);
  }
  mbar_wait(&bar_done, 0);
  tc_fence_after_sync();
  for (uint32_t c0 = 0; c0 < prm.n; c0 += 16) {
    uint32_t v[16];
    tmem_ld16(tmem_base + ((32u * warp) << 16) + c0, v);
    tmem_ld_wait();
#pragma unroll
    for (uint32_t c = 0; c < 16; ++c) d_out[static_cast<uint64_t>(32 * warp + lane) * prm.n + c0 + c] = static_cast<int32_t>(v[c]);
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}


// Issue-rate microbenchmark (diagnostic, printed by pl2gpu_selftest_umma when PL2_UMMA_BENCH is set):
// `issuers` warps each issue `reps` back-to-back int8 UMMAs of width n into their own accumulator
// columns from garbage shared memory / tensor memory, then commit.  Reports clocks per UMMA for the
// issue loop alone and up to completion.  mode 0 = SS, 1 = TS.
__global__ void __launch_bounds__(128, 1)
umma_issue_bench_kernel(uint32_t n, uint32_t reps, uint32_t mode, uint32_t issuers, uint32_t commit_every, long long* __restrict__ out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done[4];
  __shared__ uint32_t tmem_base_slot;
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(&bar_done[i], 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_base_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;
  if (warp < issuers) {
    const uint32_t style = mode >> 1;  // 0: `if (lane == 0)` region, 1: whole warp + elect.sync
    const uint32_t ts = mode & 1;
    const uint32_t idesc = make_idesc_i8(128, n, ts == 0, true);
    const uint32_t d = tmem_base + warp * (448 / issuers);
    const uint64_t da = make_smem_desc(smem_base, 2048, 128), db = make_smem_desc(smem_base + 32768, 2048, 128);
    long long t0 = 0, t1 = 0, t2 = 0;
    if (style == 0) {
      if (lane == 0) {
        t0 = clock64();
        for (uint32_t r = 0; r < reps; ++r) {
          if (ts == 0) umma_i8_ss(d, da, db, idesc, r ? 1u : 0u);
          else umma_i8_ts(d, tmem_base + 480, db, idesc, r ? 1u : 0u);
          if (commit_every) umma_commit(&bar_done[2 + warp]);  // never waited on
        }
        t1 = clock64();
        umma_commit(&bar_done[warp]);
      }
    } else {
      t0 = clock64();
      for (uint32_t r = 0; r < reps; ++r) {
        if (elect_one_sync()) {
          if (ts == 0) umma_i8_ss(d, da, db, idesc, r ? 1u : 0u);
          else umma_i8_ts(d, tmem_base + 480, db, idesc, r ? 1u : 0u);
          if (commit_every) umma_commit(&bar_done[2 + warp]);
        }
        __syncwarp();
      }
      t1 = clock64();
      if (elect_one_sync()) umma_commit(&bar_done[warp]);
      __syncwarp();
    }
    mbar_wait(&bar_done[warp], 0);
    t2 = clock64();
    if (lane == 0) {
      out[2 * warp] = t1 - t0;
      out[2 * warp + 1] = t2 - t0;
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}

// Chip-wide int8 tensor peak (pl2gpu_int8_peak): one CTA per SM, TWO issuer warps with their own accumulator
// columns ([0,240) and [240,480)) so the tensor pipe always has an independent UMMA queued (a single issuer
// accumulating into one range measures the issue/dependency latency instead: 96.6 clk per N = 160 UMMA).
// Each issuer runs `blocks` rounds of 32 back-to-back UMMAs (M = 128, N = n, K = 32), one commit per round,
// waiting for the round before the previous one so the queue stays bounded.  Operands are whatever shared /
// tensor memory holds (timing does not depend on the data).  ts = 1: A operand from tensor memory.
__global__ void __launch_bounds__(128, 1)
umma_peak_kernel(uint32_t n, uint32_t blocks, uint32_t ts) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done[2][2];
  __shared__ uint32_t tmem_base_slot;
  const uint32_t warp = uniform_warp_idx();
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i)
      for (int j = 0; j < 2; ++j) mbar_init(&bar_done[i][j], 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_base_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;
  if (warp < 2) {
    const uint32_t tmem_u = uniform_u32(tmem_base);
    const uint32_t idesc = make_idesc_i8(128, n, ts == 0, true);
    const uint64_t da = make_smem_desc(smem_base, 2048, 128), db = make_smem_desc(smem_base + 32768, 2048, 128);
    const uint32_t d = tmem_u + warp * 240;
    for (uint32_t blk = 0; blk < blocks; ++blk) {
      const uint32_t half = blk & 1;
      if (blk >= 2) mbar_wait(&bar_done[warp][half], ((blk >> 1) - 1) & 1);
      if (elect_one_sync()) {
        if (ts == 0) {
#pragma unroll 8
          for (uint32_t r = 0; r < 32; ++r) umma_i8_ss(d, da, db, idesc, 1u);
        } else {
#pragma unroll 8
          for (uint32_t r = 0; r < 32; ++r) umma_i8_ts(d, tmem_u + 480, db, idesc, 1u);
        }
        umma_commit(&bar_done[warp][half]);
      }
      __syncwarp();
    }
    for (uint32_t half = 0; half < 2; ++half) {
      const uint32_t rounds = (blocks + 1 - half) / 2;  // commits made on this half
      if (rounds) mbar_wait(&bar_done[warp][half], (rounds - 1) & 1);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}

// ---------------- kind::mxf4 (block-scaled E2M1) probes ----------------
// Tensor-memory columns [496, 512) of every lane hold UE8M0 scale bytes of 2^0; every mxf4 probe points both SFA and
// SFB there, so no scale-factor layout is involved.  The calling warp fills its own 32 lanes.
constexpr uint32_t kMxf4ProbeSfCol = 496;
__device__ __forceinline__ void fill_unit_scales(uint32_t tmem_base, uint32_t warp) {
  const uint32_t v[8] = {kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4};
  tmem_st8(tmem_base + ((32u * warp) << 16) + kMxf4ProbeSfCol, v);
  tmem_st8(tmem_base + ((32u * warp) << 16) + kMxf4ProbeSfCol + 8, v);
}

// TS probe for kind::mxf4: A rows come from global memory ([128][k_steps * 32] bytes, 64 packed E2M1 values per
// k-step), are written to tensor memory (8 columns per k-step at column 256 + 8 ks) and multiplied with the smem B
// image (K-major, descriptor fields from prm).  d_out receives the F32 accumulator bits.
__global__ void __launch_bounds__(128, 1)
umma_probe_mxf4_ts_kernel(const uint8_t* __restrict__ a_rows, const uint8_t* __restrict__ b_img, UmmaProbeParams prm, uint32_t* __restrict__ d_out /* [128][n] */) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done;
  __shared__ uint32_t tmem_base_slot;
  const uint32_t tid = threadIdx.x;
  const uint32_t warp = uniform_warp_idx();
  const uint32_t lane = tid & 31;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  uint8_t* sm = smem + (smem_base - smem_u32(smem));
  for (uint32_t i = tid; i < prm.b_bytes; i += 128) sm[i] = b_img[i];
  if (tid == 0) {
    mbar_init(&bar_done, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_base_slot);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;
  const uint32_t row_bytes = prm.k_steps * 32;
  for (uint32_t ks = 0; ks < prm.k_steps; ++ks) {
    uint32_t v[8];
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a_rows + static_cast<uint64_t>(tid) * row_bytes + ks * 32);
#pragma unroll
    for (uint32_t c = 0; c < 8; ++c) v[c] = src[c];
    tmem_st8(tmem_base + ((32u * warp) << 16) + 256 + 8 * ks, v);
  }
  fill_unit_scales(tmem_base, warp);
  tmem_st_wait();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp == 0) {
    const uint32_t tmem_u = uniform_u32(tmem_base);
    if (elect_one_sync()) {
      for (uint32_t ks = 0; ks < prm.k_steps; ++ks) {
        const uint64_t db = make_smem_desc(smem_base + ks * prm.b_step_bytes, prm.b_lbo, prm.b_sbo);
        umma_mxf4_ts(tmem_u, tmem_u + 256 + 8 * ks, db, prm.idesc, tmem_u + kMxf4ProbeSfCol, tmem_u + kMxf4ProbeSfCol, ks ? 1u : 0u);
      }
      umma_commit(&bar_done);
    }
    __syncwarp();
  }
  mbar_wait(&bar_done, 0);
  tc_fence_after_sync();
  for (uint32_t c0 = 0; c0 < prm.n; c0 += 16) {
    uint32_t v[16];
    tmem_ld16(tmem_base + ((32u * warp) << 16) + c0, v);
    tmem_ld_wait();
#pragma unroll
    for (uint32_t c = 0; c < 16; ++c) d_out[static_cast<uint64_t>(32 * warp + lane) * prm.n + c0 + c] = v[c];
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}

// Accumulator precision probe for kind::mxf4 (M = 128, N = 16).  `base_mmas` all-ones UMMAs (every A and B value
// 1.0, so each adds 64) bring every accumulator to 64 base_mmas; five more UMMAs then add one product each: A has a
// single 1.0 (K position 0 of every row), B image j = 1..5 holds the same value at all 64 K positions of column n,
// -1 when bit j - 1 of n is set (j <= 4), +1 otherwise.  Exact accumulation ends at
// 64 base_mmas + sum_j (+-1).  B images are K-major with descriptor fields (b_lbo, b_sbo).
__global__ void __launch_bounds__(128, 1)
umma_mxf4_exact_kernel(uint32_t base_mmas, uint32_t b_lbo, uint32_t b_sbo, uint32_t* __restrict__ d_out /* [128][16] */) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done;
  __shared__ uint32_t tmem_base_slot;
  constexpr uint32_t kImg = 1024;  // one 16 x 64 E2M1 image (512 bytes) per KB
  const uint32_t tid = threadIdx.x;
  const uint32_t warp = uniform_warp_idx();
  const uint32_t lane = tid & 31;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  uint8_t* sm = smem + (smem_base - smem_u32(smem));
  for (uint32_t i = tid; i < 6 * kImg; i += 128) sm[i] = 0;
  __syncthreads();
  // row n of image j: 32 bytes in two 16-byte core-matrix rows (K chunks 0 and 1)
  for (uint32_t i = tid; i < 6 * 16 * 2; i += 128) {
    const uint32_t j = i / 32, n = (i / 2) % 16, kc = i % 2;
    const uint8_t v = (j >= 1 && j <= 4 && ((n >> (j - 1)) & 1)) ? 0xAA : 0x22;
    uint8_t* row = sm + j * kImg + kc * b_lbo + (n / 8) * b_sbo + (n % 8) * 16;
    for (uint32_t b = 0; b < 16; ++b) row[b] = v;
  }
  if (tid == 0) {
    mbar_init(&bar_done, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_base_slot);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;
  {
    const uint32_t ones[8] = {0x22222222u, 0x22222222u, 0x22222222u, 0x22222222u, 0x22222222u, 0x22222222u, 0x22222222u, 0x22222222u};
    const uint32_t unit[8] = {0x2u, 0, 0, 0, 0, 0, 0, 0};
    tmem_st8(tmem_base + ((32u * warp) << 16) + 256, ones);
    tmem_st8(tmem_base + ((32u * warp) << 16) + 264, unit);
    fill_unit_scales(tmem_base, warp);
    tmem_st_wait();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp == 0) {
    const uint32_t tmem_u = uniform_u32(tmem_base);
    const uint32_t idesc = make_idesc_mxf4(128, 16);
    const uint32_t sf = tmem_u + kMxf4ProbeSfCol;
    for (uint32_t i = 0; i < base_mmas; ++i) {
      if (elect_one_sync()) umma_mxf4_ts(tmem_u, tmem_u + 256, make_smem_desc(smem_base, b_lbo, b_sbo), idesc, sf, sf, i ? 1u : 0u);
      __syncwarp();
    }
    if (elect_one_sync()) {
      for (uint32_t j = 1; j <= 5; ++j) umma_mxf4_ts(tmem_u, tmem_u + 264, make_smem_desc(smem_base + j * kImg, b_lbo, b_sbo), idesc, sf, sf, 1u);
      umma_commit(&bar_done);
    }
    __syncwarp();
  }
  mbar_wait(&bar_done, 0);
  tc_fence_after_sync();
  uint32_t v[16];
  tmem_ld16(tmem_base + ((32u * warp) << 16), v);
  tmem_ld_wait();
#pragma unroll
  for (uint32_t c = 0; c < 16; ++c) d_out[(32 * warp + lane) * 16 + c] = v[c];
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}

// Chip-wide kind::mxf4 peak (pl2gpu_mxf4_peak): as umma_peak_kernel's TS form - one CTA per SM, two issuer warps
// with accumulators [0,240) and [240,480), rounds of 32 UMMAs (M = 128, N = n, K = 64, A from tensor memory at
// column 480) - with unit scales at [496,512).  Operand values do not affect the timing.
__global__ void __launch_bounds__(128, 1)
umma_mxf4_peak_kernel(uint32_t n, uint32_t blocks) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done[2][2];
  __shared__ uint32_t tmem_base_slot;
  const uint32_t warp = uniform_warp_idx();
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i)
      for (int j = 0; j < 2; ++j) mbar_init(&bar_done[i][j], 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_base_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_slot;
  fill_unit_scales(tmem_base, warp);
  tmem_st_wait();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp < 2) {
    const uint32_t tmem_u = uniform_u32(tmem_base);
    const uint32_t idesc = make_idesc_mxf4(128, n);
    const uint64_t db = make_smem_desc(smem_base + 32768, 256, 128);
    const uint32_t d = tmem_u + warp * 240;
    const uint32_t sf = tmem_u + kMxf4ProbeSfCol;
    for (uint32_t blk = 0; blk < blocks; ++blk) {
      const uint32_t half = blk & 1;
      if (blk >= 2) mbar_wait(&bar_done[warp][half], ((blk >> 1) - 1) & 1);
      if (elect_one_sync()) {
#pragma unroll 8
        for (uint32_t r = 0; r < 32; ++r) umma_mxf4_ts(d, tmem_u + 480, db, idesc, sf, sf, 1u);
        umma_commit(&bar_done[warp][half]);
      }
      __syncwarp();
    }
    for (uint32_t half = 0; half < 2; ++half) {
      const uint32_t rounds = (blocks + 1 - half) / 2;
      if (rounds) mbar_wait(&bar_done[warp][half], (rounds - 1) & 1);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace pl2
