"""The sample-major copy's bit order (mxf4_copy_bits) and its decode (decode_mxf4) give, for every genotype code at
every position of a word, the T / H / S plane values of kTabHet / kTabHom / kTabSgn as E2M1 nibbles, in variant
order.  Both are __host__ __device__ in geno_expand.cuh; a small host program built with nvcc sweeps all 2^16 codes
of eight variants on each half of a word.  No GPU is needed."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "plink_ng_b200", "csrc")

PROGRAM = r"""
#include <cstdio>
#include "geno_expand.cuh"
using namespace pl2;

// E2M1 nibble -> value (0x0 / 0x8 are +-0, 0x2 is 1.0, 0xA is -1.0); anything else is an error.
static int e2m1_value(uint32_t nib, bool* ok) {
  switch (nib) {
    case 0x0: case 0x8: return 0;
    case 0x2: return 1;
    case 0xA: return -1;
    default: *ok = false; return 0;
  }
}
static int table_value(uint32_t table, uint32_t code) { return static_cast<int8_t>((table >> (8 * code)) & 0xFF); }

int main() {
  long bad = 0, checked = 0;
  for (uint32_t x = 0; x < (1u << 16); ++x) {
    // the 8 codes of x fill variants 0..7 in one pass and 8..15 in the other; the other half runs through
    // a different pattern (x * 40503 is a permutation of 16-bit values)
    const uint32_t y = (x * 40503u) & 0xFFFFu;
    for (int pass = 0; pass < 2; ++pass) {
      uint32_t code[16];
      for (uint32_t j = 0; j < 8; ++j) {
        code[j] = ((pass ? y : x) >> (2 * j)) & 3u;
        code[8 + j] = ((pass ? x : y) >> (2 * j)) & 3u;
      }
      uint32_t w = 0;
      for (uint32_t j = 0; j < 16; ++j) w |= mxf4_copy_bits(code[j], j);
      const Nib3 n = decode_mxf4(w);
      for (uint32_t j = 0; j < 16; ++j) {
        const uint32_t word = j / 8, sh = 4 * (j % 8);
        bool ok = true;
        const int t = e2m1_value((n.het[word] >> sh) & 0xF, &ok);
        const int h = e2m1_value((n.hom[word] >> sh) & 0xF, &ok);
        const int s = e2m1_value((n.sgn[word] >> sh) & 0xF, &ok);
        ++checked;
        if (!ok || t != table_value(kTabHet, code[j]) || h != table_value(kTabHom, code[j]) || s != table_value(kTabSgn, code[j])) {
          if (bad < 10) printf("mismatch: x=%04x pass %d variant %u code %u -> T %d H %d S %d\n", x, pass, j, code[j], t, h, s);
          ++bad;
        }
      }
    }
  }
  // an all-zero copy (out-of-range fill) is all missing: every plane 0
  const Nib3 z = decode_mxf4(0u);
  for (int i = 0; i < 2; ++i) bad += (z.het[i] | z.hom[i] | z.sgn[i]) != 0;
  printf("checked %ld, bad %ld\n", checked, bad);
  return bad != 0;
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def test_decode_mxf4_matches_plane_tables(tmp_path):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found (the library build needs it too)")
    src = tmp_path / "decode_check.cu"
    src.write_text(PROGRAM)
    exe = tmp_path / "decode_check"
    subprocess.run([nvcc, "-std=c++17", "-O1", "-I", CSRC, "-o", str(exe), str(src)], check=True, capture_output=True, text=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"checked {2 * 16 * (1 << 16)}, bad 0" in r.stdout
