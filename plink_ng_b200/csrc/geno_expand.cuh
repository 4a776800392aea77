// geno_expand.cuh - 2-bit genotype -> int8 operand expansion shared by every tensor-path kernel.
//
// A 32-bit word holds 16 consecutive samples of ONE variant (PgrGet layout).  For a plane whose
// value depends only on the genotype code, the 16 output bytes come from four PRMT (byte permute)
// instructions whose selector nibbles are the genotype codes themselves and whose source register
// is the plane's 4-entry table {value(code0), value(code1), value(code2), value(code3)}.
// Even and odd samples are handled separately (their codes are already nibble-aligned after one
// mask), so byte position p of the 16-byte result holds sample PosToSample(p) (common.cuh).
#pragma once
#include <cstdint>

namespace pl2 {

struct Sel4 {
  uint32_t e_lo, e_hi, o_lo, o_hi;  // selectors: samples {0,2,4,6}, {8,10,12,14}, {1,3,5,7}, {9,..,15}
};

__device__ __forceinline__ Sel4 make_selectors(uint32_t w) {
  const uint32_t ev = w & 0x33333333u;
  const uint32_t od = (w >> 2) & 0x33333333u;
  Sel4 s;
  s.e_lo = ev;
  s.e_hi = ev >> 16;
  s.o_lo = od;
  s.o_hi = od >> 16;
  return s;
}

__device__ __forceinline__ uint4 expand16(uint32_t table, const Sel4& s) {
  uint4 r;
  r.x = __byte_perm(table, 0u, s.e_lo);
  r.y = __byte_perm(table, 0u, s.e_hi);
  r.z = __byte_perm(table, 0u, s.o_lo);
  r.w = __byte_perm(table, 0u, s.o_hi);
  return r;
}

// Plane tables, byte c = value for genotype code c (0 hom-REF, 1 het, 2 hom-ALT, 3 missing).
constexpr uint32_t kTabHet = 0x00000100u;     // T: het indicator
constexpr uint32_t kTabHom = 0x00010001u;     // H: hom indicator (the reference's `hom` plane)
constexpr uint32_t kTabSgn = 0x00FF0001u;     // S: +1 hom-REF, -1 hom-ALT, 0 otherwise
constexpr uint32_t kTabDosage = 0x00020100u;  // g: ALT dosage 0/1/2, missing -> 0
constexpr uint32_t kTabNonmiss = 0x00010101u; // m: non-missing indicator
constexpr uint32_t kTabMiss = 0x01000000u;    // mu: missing indicator

// A plane table as a PER-THREAD register.  PRMT needs its table operand in a vector register; a
// compile-time constant gets hoisted into a uniform register and re-materialised with one extra
// IMAD.U32 in front of EVERY PRMT (164 of them in king_ts_kernel, ~25 % of its issue slots).  OR-ing in
// `thread_zero` - a value that is 0 at run time but that ptxas can prove neither constant nor
// warp-uniform (callers pass threadIdx.x * (a kernel argument >> 31)) - keeps each table in one
// vector register for the whole kernel.
__device__ __forceinline__ uint32_t table_reg(uint32_t table, uint32_t thread_zero) { return table | thread_zero; }

// ---- 2-bit genotype -> E2M1 nibble planes (kind::mxf4 operands) ----
// Every plane value is 0, +1 or -1, exact in E2M1 (1.0 = 0x2, -1.0 = 0xA, and 0x8 = -0.0).  The kind::mxf4 kernels
// read a sample-major copy (geno_tile_samples_kernel) whose bits are laid out so that the per-tile decode is a few
// masks: every tile decodes every word again, about a thousand times more often than the copy is written.
//
// A word of the copy holds 16 variants v + 0..15 of one sample.  Each variant is a pair (p, q) with
//   p = 1 for hom-REF and hom-ALT (the H plane; the magnitude of the S plane),
//   q = 1 for het and hom-ALT (the sign bit of the S plane),
// so code 0 -> (1, 0), 1 -> (0, 1), 2 -> (1, 1), 3 (missing, padding) -> (0, 0): an all-zero copy is all missing.
// Nibble i holds variant v + i in bits 1 (p) and 3 (q), and variant v + 8 + i in bits 0 (p) and 2 (q).  Then
//   S = W & 0xAAAAAAAA   (hom-REF 0x2 = +1, hom-ALT 0xA = -1, het 0x8 = -0, missing 0)
//   H = W & 0x22222222,  T = ~W & (W >> 2) & 0x22222222   (het = q and not p)
// for variants v + 0..7, and the same on W << 1 for variants v + 8..15: 9 instructions per 16 variants.
__host__ __device__ constexpr uint32_t mxf4_copy_bits(uint32_t code, uint32_t j) {  // variant j (0..15) of a word
  const uint32_t p = ~code & 1u, q = (code ^ (code >> 1)) & 1u;
  const uint32_t sh = 4 * (j & 7) + (j < 8 ? 1 : 0);
  return (p << sh) | (q << (sh + 2));
}
// One word of the copy -> two words of 8 E2M1 nibbles per plane: word 0 = variants v + 0..7, word 1 = v + 8..15,
// nibble i = variant v + i or v + 8 + i (low nibble first), i.e. K order = variant order.  Both operands of every
// product go through this function.
struct Nib3 {
  uint32_t het[2], hom[2], sgn[2];  // planes T, H, S with the values of kTabHet / kTabHom / kTabSgn
};
__host__ __device__ __forceinline__ Nib3 decode_mxf4(uint32_t w) {
  constexpr uint32_t kMag = 0x22222222u, kMagSign = 0xAAAAAAAAu;
  Nib3 r;
  const uint32_t w1 = w << 1;
  r.sgn[0] = w & kMagSign;
  r.hom[0] = w & kMag;
  r.het[0] = ~w & (w >> 2) & kMag;
  r.sgn[1] = w1 & kMagSign;
  r.hom[1] = w1 & kMag;
  r.het[1] = ~w1 & (w >> 1) & kMag;
  return r;
}

// MN-major, no-swizzle UMMA operand tile ("interleave" canonical layout,
// cute/atom/mma_traits_sm100.hpp:171): 16 consecutive samples of one variant are one 16-byte row
// of an 8-row core matrix (8 consecutive variants, 128 contiguous bytes); core matrices step by
// kCoreBytes along the sample (M/N) direction and by `lbo` along the variant (K) direction.
constexpr uint32_t kCoreBytes = 128;
__host__ __device__ constexpr uint32_t operand_lbo(uint32_t samples_in_supertile) { return (samples_in_supertile / 16) * kCoreBytes; }
__host__ __device__ constexpr uint32_t operand_offset(uint32_t k, uint32_t sample_group16, uint32_t lbo) {
  return (k >> 3) * lbo + sample_group16 * kCoreBytes + (k & 7) * 16;
}

}  // namespace pl2
