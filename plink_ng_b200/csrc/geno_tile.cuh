// geno_tile.cuh - operand re-tiling for the "TS" tensor kernels (king_ts_kernel.cuh, grm_ts_kernel.cuh):
// 128-row x 80-column pair tiles, row operand expanded into tensor memory, column operand into
// shared memory.  Kernels are static (header is included by several translation units).
#pragma once
#include "common.cuh"
#include "geno_expand.cuh"

namespace pl2 {

// 128 x 80 pair tiles.  Narrower tiles (128 x 64, eight row-operand slots instead of four) were measured and are
// SLOWER (26.7 vs 24.2 ms per 16,384 x 65,536 batch): every k-step pays ~12 KB of tcgen05.st into tensor memory
// (256 B/clk, ~48 clk) on top of its UMMA time whatever the tile width, so the widest tile that still leaves room
// for a slot ring wins (profiles/r02_king_tile_width.md).
constexpr uint32_t kTsCols = 80;
constexpr uint32_t kTsSamplePad = 640;  // lcm(128, 80)
constexpr uint32_t kTsKcJ = 64;         // variants per shared-memory stage (two k-steps)
constexpr uint32_t kTsRawBoxBytes = 32; // inner extent of the TMA box over the raw block (>= 20 bytes = 80 samples, multiple of 16)

// ---- operand re-tiling of the staged block raw[variant][pitch] (2-bit, variant-major) -------------
// Sample-major copies make every producer load of the TS kernels a contiguous run of bytes (the first
// TS version read 8 bytes per lane from 32 different rows: 336 L1 wavefronts per k-step, LSU-bound).
//
// GRM / PCA row side (int8 k-steps of 32 variants):  raw_i[row tile rt][k-step ks][row 0..127][8 bytes]   8 bytes = 32 variants of one sample
// One CTA = 64 variants x 64 samples through a shared-memory byte tile.
// Only samples [s_base, s_base + 64 * gridDim.y) are written (a job re-tiles its own row tiles only);
// row tile s_base / 128 is stored at index 0.
static __global__ void __launch_bounds__(256) geno_tile_rows_kernel(const uint8_t* __restrict__ raw, uint32_t pitch, uint32_t kstep_ct, uint32_t s_base, uint8_t* __restrict__ raw_i) {
  __shared__ uint8_t tile[64][68];
  const uint32_t v0 = blockIdx.x * 64, s0 = s_base + blockIdx.y * 64;
  const uint32_t t = threadIdx.x;
  {
    const uint32_t v = t >> 2, sw = t & 3;
    const uint32_t w = *reinterpret_cast<const uint32_t*>(raw + static_cast<uint64_t>(v0 + v) * pitch + s0 / 4 + 4 * sw);
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j) tile[v][16 * sw + j] = static_cast<uint8_t>((w >> (2 * j)) & 3u);
  }
  __syncthreads();
  {
    const uint32_t sl = t >> 2, vw = t & 3;
    uint32_t w = 0;
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j) w |= static_cast<uint32_t>(tile[16 * vw + j][sl]) << (2 * j);
    const uint32_t s = s0 + sl, v = v0 + 16 * vw;
    *reinterpret_cast<uint32_t*>(raw_i + (static_cast<uint64_t>((s - s_base) >> 7) * kstep_ct + (v >> 5)) * 1024 + (s & 127) * 8 + 4 * ((v >> 4) & 1)) = w;
  }
}

// Sample-major copy for 64-variant k-steps (king_ts_kernel.cuh):  raw_x[k-step ks][sample s][16 bytes]
// 16 bytes = 64 variants of one sample; word j / 16 holds variant 64 ks + j in the decode-friendly bit order of
// geno_expand.cuh (mxf4_copy_bits: variant j % 16 < 8 in bits 1 and 3 of nibble j % 8, else in bits 0 and 2).
// Samples [0, gridDim.y * 64) are written; one CTA = 64 variants x 64 samples through a shared-memory byte tile.
static __global__ void __launch_bounds__(256) geno_tile_samples_kernel(const uint8_t* __restrict__ raw, uint32_t pitch, uint32_t sample_ct_x, uint8_t* __restrict__ raw_x) {
  __shared__ uint8_t tile[64][68];
  const uint32_t v0 = blockIdx.x * 64, s0 = blockIdx.y * 64;
  const uint32_t t = threadIdx.x;
  {
    const uint32_t v = t >> 2, sw = t & 3;
    const uint32_t w = *reinterpret_cast<const uint32_t*>(raw + static_cast<uint64_t>(v0 + v) * pitch + s0 / 4 + 4 * sw);
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j) tile[v][16 * sw + j] = static_cast<uint8_t>((w >> (2 * j)) & 3u);
  }
  __syncthreads();
  {
    const uint32_t sl = t >> 2, vw = t & 3;
    uint32_t w = 0;
#pragma unroll
    for (uint32_t j = 0; j < 16; ++j) w |= mxf4_copy_bits(tile[16 * vw + j][sl], j);
    *reinterpret_cast<uint32_t*>(raw_x + (static_cast<uint64_t>(blockIdx.x) * sample_ct_x + s0 + sl) * 16 + 4 * vw) = w;
  }
}

}  // namespace pl2
