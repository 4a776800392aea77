// king_ts_kernel.cuh - KING pair counts, "TS" tensor kernel on block-scaled FP4 UMMAs (tcgen05.mma kind::mxf4):
// the row-side (A) operand is expanded into tensor memory (tcgen05.st), the column-side (B) operand into shared
// memory, both from the same sample-major copy of the genotype block (geno_tile_samples_kernel).
//
// Why FP4 is exact here: every operand value is 0, +1 or -1 (E2M1 0x0 / 0x2 / 0xA), every scale byte is 2^0 (UE8M0
// 0x7F), so each product is the integer product, and every partial sum is an integer of magnitude at most the
// variant count of one launch (<= kMaxStageVariantsEx = 2^20), which the F32 accumulator holds exactly below 2^24
// (pl2gpu_selftest_umma checks this on the device past 2^20).  The epilogue converts back to int32 with
// cvt.rni.s32.f32, so the HBM accumulators and everything downstream stay int32.  kind::mxf4 runs at twice the
// kind::i8 rate, and a k-step covers 64 variants instead of 32 for the same tensor-memory store cost.
//
// Tile = 128 rows x 80 cols.  TMEM columns: [0,400) F32 accumulators TT|TH, HT|HH, SS, [400,496) four A slots of
// 24 columns (planes T, H, S; 8 columns = 64 packed E2M1 per lane), [496,512) unit scale bytes: SFA and SFB of
// every UMMA point there, so no scale-factor layout is involved.
//
// Operand staging: one producer warp feeds two shared-memory rings with 3-D TMA copies of the sample-major copy,
// four k-steps per copy: the row tile's [4][128][16 B] and the column tile's [4][80][16 B].  The expansion warps
// read their 16-byte runs with conflict-free LDS.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "geno_expand.cuh"
#include "geno_tile.cuh"
#include "umma.cuh"

namespace pl2 {

// F32 accumulation is exact for integers below 2^24, and no partial sum of a launch exceeds its variant count.
static_assert(kMaxStageVariantsEx <= (1u << 24), "king_ts_kernel accumulates in F32: a launch must stay below 2^24 variants");

constexpr uint32_t kTsKstep = 64;              // variants per k-step (K of one kind::mxf4 UMMA)
constexpr uint32_t kTsGroupsJ = kTsCols / 16;  // 16-column chunks per accumulator plane (epilogue)
constexpr uint32_t kTsAccCols = 5 * kTsCols;   // 400
constexpr uint32_t kTsTileAccWords = kTsAccCols * kTileRows;
constexpr uint32_t kTsASlots = 4;
constexpr uint32_t kTsASlotCols = 24;
constexpr uint32_t kTsSfCol = kTsAccCols + kTsASlots * kTsASlotCols;  // 496
static_assert(kTsSfCol + 16 <= 512, "TMEM budget: accumulators + A slots + scale columns");
// B stage (one k-step), K-major no-swizzle: a core matrix is 8 samples x 16 bytes (32 K).  K chunk kc (0, 1) holds
// the 30 eight-sample groups [T 0..9 | H 0..9 | S 0..9] at kCoreBytes apart; the +64 makes the two chunks' rows
// fall in different bank halves, so the column warps' 8-byte stores are conflict-free.  The column warps and the
// issuer hand the stages over two k-steps at a time (one wait, fence and arrive per two k-steps); deeper stages
// would not leave room for two CTAs per SM.
constexpr uint32_t kTsStagesJ = 4;
constexpr uint32_t kTsHandJ = 2;                  // k-steps per B-stage handshake
constexpr uint32_t kTsBarsJ = kTsStagesJ / kTsHandJ;
constexpr uint32_t kTsLboJ = 3 * (kTsCols / 8) * kCoreBytes + 64;  // 3904: K-chunk stride
constexpr uint32_t kTsStageBytesJ = 2 * kTsLboJ;                    // 7808
constexpr uint32_t kTsRingKsteps = 4;                              // k-steps per TMA copy (one ring slot)
constexpr uint32_t kTsRawJSlots = 4;
constexpr uint32_t kTsRawJBytes = kTsRingKsteps * kTsCols * 16;    // 5120
constexpr uint32_t kTsRawISlots = 4;
constexpr uint32_t kTsRawIBytes = kTsRingKsteps * kTileRows * 16;  // 8192
constexpr uint32_t kTsSmemOffRawI = (kTsStagesJ * kTsStageBytesJ + 1023u) & ~1023u;  // 31744
constexpr uint32_t kTsSmemOffRawJ = kTsSmemOffRawI + kTsRawISlots * kTsRawIBytes;
constexpr uint32_t kTsSmemBytes = kTsSmemOffRawJ + kTsRawJSlots * kTsRawJBytes + 1024;
constexpr uint32_t kTsRowWarps = 8;
constexpr uint32_t kTsColWarps = kTsCols / 8;  // 10: warp = one 8-sample group, lane = (sample, 16-variant word)
constexpr uint32_t kTsIssuerWarp = kTsRowWarps + kTsColWarps;
constexpr uint32_t kTsLoaderWarp = kTsIssuerWarp + 1;
constexpr uint32_t kTsThreads = 32 * (kTsRowWarps + kTsColWarps + 2);  // + the UMMA issuer warp + the TMA producer warp
static_assert(kTsSmemOffRawJ % 128 == 0 && kTsRawJBytes % 128 == 0, "TMA destination alignment");

__global__ void __launch_bounds__(kTsThreads, 1)
king_ts_kernel(const __grid_constant__ CUtensorMap tmap_i, const __grid_constant__ CUtensorMap tmap_j, uint32_t variant_ct_padded /* multiple of 256 */, const uint32_t* __restrict__ tile_order, const uint32_t* __restrict__ tile_rt, const uint32_t* __restrict__ tile_tc, int32_t* __restrict__ raw_acc) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_full_a[kTsASlots];
  __shared__ __align__(8) uint64_t bar_empty_a[kTsASlots];
  __shared__ __align__(8) uint64_t bar_full_b[kTsBarsJ];
  __shared__ __align__(8) uint64_t bar_empty_b[kTsBarsJ];
  __shared__ __align__(8) uint64_t bar_full_rj[kTsRawJSlots];
  __shared__ __align__(8) uint64_t bar_empty_rj[kTsRawJSlots];
  __shared__ __align__(8) uint64_t bar_full_ri[kTsRawISlots];
  __shared__ __align__(8) uint64_t bar_empty_ri[kTsRawISlots];
  __shared__ __align__(8) uint64_t bar_acc;
  __shared__ uint32_t tmem_base_slot;

  const uint32_t tid = threadIdx.x;
  const uint32_t warp = uniform_warp_idx();
  const uint32_t lane = tid & 31;
  const uint32_t tile = tile_order[blockIdx.x];
  const uint32_t rt = tile_rt[tile];
  const uint32_t ct = tile_tc[tile];
  const uint32_t ksteps = variant_ct_padded / kTsKstep;  // multiple of 4
  const uint32_t slot_iters = ksteps / kTsRingKsteps;
  const uint32_t smem_base = (smem_u32(smem) + 1023u) & ~1023u;

  if (tid == 0) {
    for (uint32_t s = 0; s < kTsASlots; ++s) {
      mbar_init(&bar_full_a[s], 4);             // one arrival per row-side warp of the owning group
      mbar_init(&bar_empty_a[s], 1);
    }
    for (uint32_t s = 0; s < kTsBarsJ; ++s) {
      mbar_init(&bar_full_b[s], kTsColWarps);
      mbar_init(&bar_empty_b[s], 1);
    }
    for (uint32_t s = 0; s < kTsRawJSlots; ++s) {
      mbar_init(&bar_full_rj[s], 1);            // the producer's expect_tx arrival
      mbar_init(&bar_empty_rj[s], kTsColWarps);
    }
    for (uint32_t s = 0; s < kTsRawISlots; ++s) {
      mbar_init(&bar_full_ri[s], 1);
      mbar_init(&bar_empty_ri[s], kTsRowWarps); // every row warp reads two of the slot's four k-steps
    }
    mbar_init(&bar_acc, 1);
    mbar_fence_init();
  }
  __syncthreads();  // barriers initialised
  // Tensor memory is needed by the row warps and the issuer only.  The allocation blocks while the previous CTA on
  // this SM still holds its 512 columns (two CTAs fit an SM otherwise), so the TMA producer and the column warps do
  // NOT wait for it: rings and B stages of this tile fill up behind the previous tile's epilogue.
  uint32_t tmem_base = 0;
  if (warp == kTsIssuerWarp) tmem_alloc<512>(&tmem_base_slot);
  if (warp < kTsRowWarps || warp == kTsIssuerWarp) {
    tc_fence_before_sync();
    named_bar_sync<1, 32 * (kTsRowWarps + 1)>();
    tc_fence_after_sync();
    tmem_base = tmem_base_slot;
  }

  if (warp < kTsRowWarps) {
    // ---------------- row-side producers: 2-bit codes -> E2M1 nibbles -> tensor memory ----------------
    // Two groups of four warps (group = warp / 4); group g owns k-steps ks = 2 n + g and the A slots
    // ks % 4 in {g, g + 2}.  Thread = TMEM lane = sample 128 rt + 32 (warp % 4) + lane.  The codes of
    // the next k-step are expanded while the UMMAs of the previous ones run.
    const uint32_t grp = warp >> 2;
    const uint32_t lq = warp & 3;
    const uint32_t row = 32 * lq + lane;
    const uint32_t ring_i = smem_base + kTsSmemOffRawI + row * 16;
    const uint32_t taddr_lane = tmem_base + ((32u * lq) << 16);
    if (grp == 0) {
      // unit scales for every UMMA of the tile; ordered before the first A slot's arrival by the wait::st below
      const uint32_t one[8] = {kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4, kUe8m0One4};
      tmem_st8(taddr_lane + kTsSfCol, one);
      tmem_st8(taddr_lane + kTsSfCol + 8, one);
    }
    struct ExpI {
      uint32_t v[3][8];
    };
    auto expand_i = [&](const uint4& w) -> ExpI {
      ExpI e;
      const uint32_t words[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const Nib3 n = decode_mxf4(words[i]);
        e.v[0][2 * i] = n.het[0]; e.v[0][2 * i + 1] = n.het[1];
        e.v[1][2 * i] = n.hom[0]; e.v[1][2 * i + 1] = n.hom[1];
        e.v[2][2 * i] = n.sgn[0]; e.v[2][2 * i + 1] = n.sgn[1];
      }
      return e;
    };
    // One ring slot = k-steps 4 q .. 4 q + 3; this group needs 4 q + grp and 4 q + grp + 2.  Both runs are read
    // (and the slot released) up front, expanded one k-step ahead of the tensor-memory store.
    struct Words {
      uint4 w[2];
    };
    auto load_slot = [&](uint32_t q) -> Words {
      const uint32_t si = q % kTsRawISlots;
      mbar_wait(&bar_full_ri[si], (q / kTsRawISlots) & 1);
      Words r;
      r.w[0] = lds128(ring_i + si * kTsRawIBytes + grp * (kTileRows * 16));
      r.w[1] = lds128(ring_i + si * kTsRawIBytes + (grp + 2) * (kTileRows * 16));
      return r;  // the slot is released only after both runs have gone through tcgen05.st (see below)
    };
    Words words = load_slot(0);
    ExpI cur = expand_i(words.w[0]);
    static_assert(kTsASlots == kTsRingKsteps, "k-step 4 q + grp + 2 h always uses A slot grp + 2 h");
    for (uint32_t q = 0; q < slot_iters; ++q) {
#pragma unroll
      for (uint32_t h = 0; h < 2; ++h) {
        const uint32_t slot = grp + 2 * h;  // used for the q-th time
        mbar_wait(&bar_empty_a[slot], (q & 1) ^ 1);
        tc_fence_after_sync();
        const uint32_t ta = taddr_lane + kTsAccCols + slot * kTsASlotCols;
        tmem_st8(ta, cur.v[0]);
        tmem_st8(ta + 8, cur.v[1]);
        tmem_st8(ta + 16, cur.v[2]);
        tmem_st_wait();
        tc_fence_before_sync();
        mbar_arrive_warp(&bar_full_a[slot], lane);
        if (h == 0) {
          cur = expand_i(words.w[1]);
        } else {
          // Release the ring slot HERE: the warp-collective tcgen05.st above could only issue once every lane's
          // expanded registers - hence both ld.shared results - were complete (umma.cuh, mbar_arrive_warp).
          mbar_arrive_warp(&bar_empty_ri[q % kTsRawISlots], lane);
          if (q + 1 < slot_iters) {
            words = load_slot(q + 1);
            cur = expand_i(words.w[0]);
          }
        }
      }
    }
  } else if (warp < kTsIssuerWarp) {
    // ---------------- column-side producers: 2-bit codes -> E2M1 nibbles in shared memory ----------------
    // Warp j = samples 8 j .. 8 j + 7 of the tile (core-matrix group j); lane = (sample 8 j + lane / 4, 16-variant
    // word w = lane % 4).  Word w of a k-step is K bytes 8 w .. 8 w + 7 of the sample's 32-byte row: K chunk w / 2,
    // byte (w % 2) * 8 of its 16-byte core-matrix row - the same K order as the row side's TMEM columns 2 w, 2 w + 1.
    const uint32_t j = warp - kTsRowWarps;
    const uint32_t n = 8 * j + (lane >> 2);
    const uint32_t w = lane & 3;
    const uint32_t ring_j = smem_base + kTsSmemOffRawJ + n * 16 + 4 * w;
    const uint32_t dst = (w >> 1) * kTsLboJ + j * kCoreBytes + (n & 7) * 16 + (w & 1) * 8;
    constexpr uint32_t kPlaneOff = (kTsCols / 8) * kCoreBytes;  // T -> H -> S
    for (uint32_t q = 0; q < slot_iters; ++q) {
      const uint32_t sj = q % kTsRawJSlots;
      mbar_wait(&bar_full_rj[sj], (q / kTsRawJSlots) & 1);
      uint32_t words[kTsRingKsteps];
#pragma unroll
      for (uint32_t kk = 0; kk < kTsRingKsteps; ++kk) words[kk] = lds32(ring_j + sj * kTsRawJBytes + kk * (kTsCols * 16));
      static_assert(kTsRingKsteps == kTsStagesJ, "one ring slot fills the B stages once");
#pragma unroll
      for (uint32_t sb = 0; sb < kTsStagesJ; ++sb) {
        const uint32_t hb = sb / kTsHandJ;
        const Nib3 e = decode_mxf4(words[sb]);
        if (sb % kTsHandJ == 0) mbar_wait(&bar_empty_b[hb], (q & 1) ^ 1);
        const uint32_t a0 = smem_base + sb * kTsStageBytesJ + dst;
        sts64x2(a0, e.het[0], e.het[1]);
        sts64x2(a0 + kPlaneOff, e.hom[0], e.hom[1]);
        sts64x2(a0 + 2 * kPlaneOff, e.sgn[0], e.sgn[1]);
        if (sb % kTsHandJ == kTsHandJ - 1) {
          fence_proxy_async_smem();
          mbar_arrive_warp(&bar_full_b[hb], lane);
        }
      }
      mbar_arrive_warp(&bar_empty_rj[sj], lane);  // every word went into an st.shared above
    }
  } else if (warp == kTsIssuerWarp) {
    // ---------------- UMMA issuer: whole warp loops, one elected lane issues (umma.cuh) ----------------
    // One outer iteration = the 4 shared-memory stages = 4 k-steps = one round of the 4 A slots, so every slot
    // index, parity and descriptor offset is a compile-time constant.
    static_assert(kTsStagesJ == 4 && kTsASlots == 4, "issuer unrolling assumes 4 stages / 4 slots");
    constexpr uint32_t idesc_n160 = make_idesc_mxf4(128, 2 * kTsCols);
    constexpr uint32_t idesc_n80 = make_idesc_mxf4(128, kTsCols);
    const uint32_t tmem_u = uniform_u32(tmem_base);
    const uint32_t sf = tmem_u + kTsSfCol;
    const uint64_t desc0 = make_smem_desc(smem_base, kTsLboJ, kCoreBytes);
    for (uint32_t it0 = 0; it0 < ksteps; it0 += kTsStagesJ) {
      const uint32_t ph = (it0 / kTsStagesJ) & 1;
#pragma unroll
      for (uint32_t sb = 0; sb < kTsStagesJ; ++sb) {
        if (sb % kTsHandJ == 0) mbar_wait(&bar_full_b[sb / kTsHandJ], ph);
        mbar_wait(&bar_full_a[sb], ph);
        tc_fence_after_sync();
        if (elect_one_sync()) {
          const uint32_t acc = (it0 | sb) ? 1u : 0u;
          const uint64_t b_th = desc0 + ((sb * kTsStageBytesJ) >> 4);
          const uint64_t b_s = b_th + ((2 * (kTsCols / 8) * kCoreBytes) >> 4);
          const uint32_t ta = tmem_u + kTsAccCols + sb * kTsASlotCols;
          umma_mxf4_ts(tmem_u + 0, ta, b_th, idesc_n160, sf, sf, acc);
          umma_mxf4_ts(tmem_u + 2 * kTsCols, ta + 8, b_th, idesc_n160, sf, sf, acc);
          umma_mxf4_ts(tmem_u + 4 * kTsCols, ta + 16, b_s, idesc_n80, sf, sf, acc);
          umma_commit(&bar_empty_a[sb]);
          if (sb % kTsHandJ == kTsHandJ - 1) umma_commit(&bar_empty_b[sb / kTsHandJ]);
        }
        __syncwarp();
      }
    }
    if (elect_one_sync()) umma_commit(&bar_acc);
    __syncwarp();
  } else {
    // ---------------- TMA producer: one elected lane keeps both raw rings full ----------------
    if (elect_one_sync()) {
      const uint32_t ring_j = smem_base + kTsSmemOffRawJ, ring_i = smem_base + kTsSmemOffRawI;
      const int32_t row0 = static_cast<int32_t>(rt * kTileRows), col0 = static_cast<int32_t>(ct * kTsCols);
      for (uint32_t q = 0; q < slot_iters; ++q) {
        const int32_t ks0 = static_cast<int32_t>(q * kTsRingKsteps);
        const uint32_t si = q % kTsRawISlots;
        mbar_wait(&bar_empty_ri[si], ((q / kTsRawISlots) & 1) ^ 1);
        mbar_expect_tx(&bar_full_ri[si], kTsRawIBytes);
        tma_load_3d(ring_i + si * kTsRawIBytes, &tmap_i, 0, row0, ks0, &bar_full_ri[si]);
        const uint32_t sj = q % kTsRawJSlots;
        mbar_wait(&bar_empty_rj[sj], ((q / kTsRawJSlots) & 1) ^ 1);
        mbar_expect_tx(&bar_full_rj[sj], kTsRawJBytes);
        tma_load_3d(ring_j + sj * kTsRawJBytes, &tmap_j, 0, col0, ks0, &bar_full_rj[sj]);
      }
    }
    __syncwarp();
  }

  if (warp < kTsRowWarps) {
    // ---------------- epilogue: TMEM -> int32 -> shared memory -> bulk reduce-add into the HBM accumulators ----------------
    // The accumulators of a tile are one contiguous int32 [5 x 80 columns][128 rows] block.  Instead of a
    // load-add-store per element from registers (latency-bound: ~16 KB in flight per SM, ~45 us per tile, i.e. >10 %
    // of the tile), each accumulator plane (80 columns = 40 KB) is staged in shared memory - the operand stages and
    // rings are idle now - and handed to the TMA unit as ONE cp.reduce.async.bulk .add.s32: the addition happens at
    // the L2, nothing is read back, and tensor memory is released as soon as the last tcgen05.ld has returned.
    mbar_wait(&bar_acc, 0);
    tc_fence_after_sync();
    constexpr uint32_t kPlaneBytes = kTsCols * kTileRows * 4;  // 40960
    static_assert(2 * kPlaneBytes <= kTsSmemBytes - 1024, "two staging planes must fit the dynamic shared memory");
    const uint32_t lq = warp & 3, half = warp >> 2;
    const uint32_t rsample = 32 * lq + lane;  // rows and columns are in natural sample order
    int32_t* acc_tile = raw_acc + static_cast<uint64_t>(tile) * kTsTileAccWords;
#pragma unroll 1
    for (uint32_t q = 0; q < 5; ++q) {  // accumulator planes TT, TH, HT, HH, SS
      const uint32_t stage = smem_base + (q & 1) * kPlaneBytes + rsample * 4;
      if (q >= 2) {
        // plane q - 2 used this staging buffer: its bulk reduction must have finished READING shared memory
        if (tid == 0) bulk_wait_group_read<1>();
        named_bar_sync<2, 32 * kTsRowWarps>();
      }
      // 5 chunks of 16 columns per plane and lane quarter: half 0 takes chunks 0, 2, 4, half 1 takes 1, 3
#pragma unroll 1
      for (uint32_t cgrp = half; cgrp < kTsGroupsJ; cgrp += 2) {
        uint32_t v[16];
        tmem_ld16(tmem_base + ((32u * lq) << 16) + 16 * (q * kTsGroupsJ + cgrp), v);
        tmem_ld_wait();
#pragma unroll
        for (uint32_t c = 0; c < 16; ++c) sts32(stage + (cgrp * 16 + c) * (kTileRows * 4), static_cast<uint32_t>(f32_bits_to_s32_rn(v[c])));
      }
      fence_proxy_async_smem();
      if (q == 4) tc_fence_before_sync();  // last tcgen05.ld of this warp is complete
      named_bar_sync<2, 32 * kTsRowWarps>();
      if (tid == 0) {
        bulk_reduce_add_s32(acc_tile + static_cast<uint64_t>(q) * (kTsCols * kTileRows), smem_base + (q & 1) * kPlaneBytes, kPlaneBytes);
        bulk_commit_group();
      }
    }
  }
  if (warp < kTsRowWarps || warp == kTsIssuerWarp) {
    // all tensor-memory reads are done: hand the columns to the next CTA before the reductions have drained
    named_bar_sync<1, 32 * (kTsRowWarps + 1)>();
    if (warp == kTsIssuerWarp) {
      tc_fence_after_sync();
      tmem_dealloc<512>(tmem_base);
    }
  }
  if (tid == 0) bulk_wait_group_read<0>();  // shared memory must outlive the reductions' reads
}

}  // namespace pl2
