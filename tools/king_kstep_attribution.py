"""Where the k-step of king_ts_kernel goes: the kernel at the bench.py shape against ablated copies of itself.

    python tools/king_kstep_attribution.py build OUT [--src TREE]   # CPU: patch copies of TREE's sources, compile
    python tools/king_kstep_attribution.py run OUT                   # GPU: time every variant built under OUT

`build` copies the package of TREE (default: this repository) once per variant to OUT/<variant>/, rewrites
king_ts_kernel.cuh there and compiles that copy's libpl2gpu.so.  The shipped library is never patched.  Variants:
  full          the kernel as it is
  umma_only     neither producer writes an operand: the UMMAs run on whatever the stages and A slots hold
  no_row_expand the row warps store the raw copy words into tensor memory instead of decoded planes
  no_col_expand the column warps store the raw copy words into shared memory instead of decoded planes
  no_row_st     the row warps decode but skip the tcgen05.st of the A operand
Every synchronisation stays, so each variant differs from `full` by the work it removes.  The patches match both the
decode of this tree (decode_mxf4) and the earlier one (expand_nibbles), so a parent checkout can be measured too.
Counts computed by a patched variant are wrong by design; only its time means something.

`run` times one launch of every variant (2 warm-up steps, then the median of 3) on 100,000 samples x 131,072 variants
with bench.py's generator, in a subprocess each, and prints one JSON line per variant with ms per launch, the SM clock
and the power seen meanwhile (bench.ClockSampler)."""
import json
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
DECODE = r"(?:decode_mxf4|expand_nibbles)"
ROW_DECODE = (DECODE + r"\(words\[i\]\)", "Nib3{{words[i], words[i]}, {words[i], words[i]}, {words[i], words[i]}}")
COL_DECODE = (DECODE + r"\(words\[(sb|kk)\]\)", r"Nib3{{words[\1], words[\1]}, {words[\1], words[\1]}, {words[\1], words[\1]}}")
ROW_ST = r"tmem_st8\(ta, cur\.v\[0\]\);\s*tmem_st8\(ta \+ 8, cur\.v\[1\]\);\s*tmem_st8\(ta \+ 16, cur\.v\[2\]\);\s*tmem_st_wait\(\);"
COL_STS = (r"sts64x2\(a0, e\.het\[0\], e\.het\[1\]\);\s*sts64x2\(a0 \+ kPlaneOff, e\.hom\[0\], e\.hom\[1\]\);\s*sts64x2\(a0 \+ 2 \* kPlaneOff, e\.sgn\[0\], e\.sgn\[1\]\);", "")
# keep the decoded registers alive without storing them
KEEP_ROW = "#pragma unroll\n        for (int p_ = 0; p_ < 3; ++p_)\n          for (int i_ = 0; i_ < 8; ++i_) asm volatile(\"\" ::\"r\"(cur.v[p_][i_]));"

VARIANTS = {
    "full": [],
    "umma_only": [(ROW_ST, ""), COL_STS],
    "no_row_expand": [ROW_DECODE],
    "no_col_expand": [COL_DECODE],
    "no_row_st": [(ROW_ST, KEEP_ROW)],
}


def build(out, src):
    kernel = os.path.join(src, "plink_ng_b200", "csrc", "king_ts_kernel.cuh")
    text = open(kernel).read()
    for name, patches in VARIANTS.items():
        dst = os.path.join(out, name)
        shutil.rmtree(dst, ignore_errors=True)
        shutil.copytree(os.path.join(src, "plink_ng_b200"), os.path.join(dst, "plink_ng_b200"), ignore=shutil.ignore_patterns("*.so", "plink2_b200", "__pycache__"))
        shutil.copytree(os.path.join(src, "include"), os.path.join(dst, "include"))
        t = text
        for pat, rep in patches:
            t, n = re.subn(pat, rep, t)
            if n != 1:
                raise SystemExit(f"{name}: pattern {pat!r} matched {n} times in {kernel}")
        open(os.path.join(dst, "plink_ng_b200", "csrc", "king_ts_kernel.cuh"), "w").write(t)
        csrc = os.path.join(dst, "plink_ng_b200", "csrc")
        cmd = [NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared", "-o", "../libpl2gpu.so",
               "pl2gpu.cu", "ld.cu", "grm.cu", "pca.cu", "score.cu", "-lcudart"]
        print(f"building {name} ...", flush=True)
        subprocess.run(cmd, cwd=csrc, check=True)


CHILD = r"""
import json, statistics, sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(1, sys.argv[2])
import torch
import plink_ng_b200 as p
from plink_ng_b200.host import KING_ALGO_TENSOR_TS, KingJob
from bench import ClockSampler, synth_genovecs
n, mb = 100_000, 131_072
row_bytes = (n + 31) // 32 * 8
dev = torch.device("cuda", 0)
geno = synth_genovecs(torch, n, 0, mb, dev)
torch.cuda.synchronize()
with p.GpuContext(0) as ctx, KingJob(ctx, n, 0, n, KING_ALGO_TENSOR_TS, max_variants_per_add=mb) as job:
    for _ in range(2):
        job.add_variants_device(geno.data_ptr(), row_bytes, mb, complete=True)
    ctx.synchronize()
    s = ClockSampler(0)
    s.start()
    ms = []
    for _ in range(3):
        job.add_variants_device(geno.data_ptr(), row_bytes, mb, complete=True)
        ctx.synchronize()
        ms.append(job.last_kernel_ms())
    clocks = s.stop()
print(json.dumps({"kernel_ms": statistics.median(ms), "kernel_ms_all": ms, "clocks": clocks, "gpu": torch.cuda.get_device_name(0)}))
"""


def run(out):
    for name in VARIANTS:
        d = os.path.join(out, name)
        if not os.path.exists(os.path.join(d, "plink_ng_b200", "libpl2gpu.so")):
            continue
        r = subprocess.run([sys.executable, "-c", CHILD, d, ROOT], capture_output=True, text=True)
        line = r.stdout.strip().splitlines()[-1] if r.returncode == 0 and r.stdout.strip() else json.dumps({"error": r.stderr[-2000:]})
        print(json.dumps({"variant": name, "tree": out, **json.loads(line)}), flush=True)


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "build":
        src = sys.argv[sys.argv.index("--src") + 1] if "--src" in sys.argv else ROOT
        build(os.path.abspath(sys.argv[2]), os.path.abspath(src))
    elif len(sys.argv) == 3 and sys.argv[1] == "run":
        run(os.path.abspath(sys.argv[2]))
    else:
        raise SystemExit(__doc__)
