"""Reference outputs of two library functions the host program restates, for tests/test_host_program.py:

  dtoa_g_p8.json    SHA-256 digest and line count of the text the reference's dtoa_g_p8
                    (2.0/include/plink2_string.cc:2641) writes, one line per input of test_host_program.dtoa_p8_inputs()
  sfmt_seed11.u32   the first 5,000 draws of the reference's SFMT-19937 (2.0/include/SFMT.c) seeded with 11

Small harnesses are compiled against the reference's headers and the objects oracle/build_ref.sh leaves in
oracle/_ref/obj.  Run from the repository root:

    python tests/golden/make_host_format_set.py <reference 2.0 source directory>
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from test_host_program import SFMT_DRAWS, dtoa_p8_inputs  # noqa: E402

OBJ = os.path.join(ROOT, "oracle", "_ref", "obj")

DTOA_HARNESS = r"""
#include <cstdio>
#include "plink2_string.h"
int main(int argc, char** argv) {
  FILE* in = fopen(argv[1], "rb"); FILE* out = fopen(argv[2], "w");
  double x; char buf[64];
  while (fread(&x, 8, 1, in) == 1) { char* e = plink2::dtoa_g_p8(x, buf); *e = 0; fprintf(out, "%s\n", buf); }
  fclose(in); fclose(out); return 0;
}
"""

SFMT_HARNESS = r"""
#include <stdio.h>
#include <stdlib.h>
#include "SFMT.h"
int main(int argc, char** argv) {
  sfmt_t s; uint32_t seed = strtoul(argv[1], 0, 10); unsigned long n = strtoul(argv[2], 0, 10);
  sfmt_init_gen_rand(&s, seed);
  FILE* f = fopen(argv[3], "wb");
  for (unsigned long k = 0; k < n; ++k) { uint32_t v = sfmt_genrand_uint32(&s); fwrite(&v, 4, 1, f); }
  fclose(f);
  return 0;
}
"""


def main(src):
    inc = os.path.join(src, "include")
    with tempfile.TemporaryDirectory() as tmp:
        h, exe = os.path.join(tmp, "dtoa.cc"), os.path.join(tmp, "dtoa")
        open(h, "w").write(DTOA_HARNESS)
        objs = [os.path.join(OBJ, "include_plink2_%s_cc.o" % x) for x in ("string", "base", "bits", "float", "simd")]
        subprocess.run(["g++", "-O1", "-std=c++11", "-mavx2", "-mbmi", "-mbmi2", "-mfma", "-mlzcnt", "-w", "-I" + inc, "-I" + os.path.join(src, "simde"), h] + objs + ["-o", exe], check=True)
        dtoa_p8_inputs().tofile(os.path.join(tmp, "in.bin"))
        subprocess.run([exe, os.path.join(tmp, "in.bin"), os.path.join(tmp, "out.txt")], check=True)
        text = open(os.path.join(tmp, "out.txt"), "rb").read()
        with open(os.path.join(HERE, "dtoa_g_p8.json"), "w") as f:
            json.dump({"lines": text.count(b"\n"), "sha256": hashlib.sha256(text).hexdigest()}, f, indent=1)
            f.write("\n")

        h, exe = os.path.join(tmp, "sfmt.c"), os.path.join(tmp, "sfmt")
        open(h, "w").write(SFMT_HARNESS)
        subprocess.run(["gcc", "-O1", "-DSFMT_MEXP=19937", "-I" + inc, h, os.path.join(OBJ, "include_SFMT_c.o"), "-lm", "-o", exe], check=True)
        subprocess.run([exe, "11", str(SFMT_DRAWS), os.path.join(HERE, "sfmt_seed11.u32")], check=True)


if __name__ == "__main__":
    main(sys.argv[1])
