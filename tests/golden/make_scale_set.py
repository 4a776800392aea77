"""Reference results for the at-scale parity tests (tests/test_scale_gpu.py, tests/test_multi_gpu.py).

Their inputs are megabytes to gigabytes, too large to keep here, so the tests regenerate them from a seed and this
script stores what the reference wrote for them: SHA-256 digests of the files the product must reproduce byte for
byte, the row counts and table filter the tests use, and a fixed sample of the fp32 GRM entries that are compared
within a tolerance.  Run from the repository root after oracle/build_ref.sh:

    python tests/golden/make_scale_set.py
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from test_scale_gpu import DATASETS, write_dataset  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "plink2")
REF_LAPACK = os.path.join(ROOT, "oracle", "_ref", "plink2_lapack")
THREADS = str(max(1, min(32, len(os.sched_getaffinity(0)))))
GRM_OFFDIAG_SAMPLE = 4096


def grm_sample_index(n):
    """Positions in the .grm.bin lower triangle: every diagonal entry and a fixed random set of the others."""
    diag = np.arange(n, dtype=np.int64) * (np.arange(n, dtype=np.int64) + 3) // 2
    rest = np.setdiff1d(np.arange(n * (n + 1) // 2, dtype=np.int64), diag)
    pick = np.random.default_rng(n).choice(rest, size=GRM_OFFDIAG_SAMPLE, replace=False)
    return np.sort(np.concatenate([diag, pick])).astype(np.uint32)


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def run(binary, pre, flags, out):
    subprocess.run([binary, "--bfile", pre] + flags + ["--threads", THREADS, "--out", out], check=True, stdout=subprocess.DEVNULL)


def grm_sample(out, n, name):
    g = np.fromfile(out + ".grm.bin", dtype=np.float32)
    assert g.size == n * (n + 1) // 2
    idx = grm_sample_index(n)
    np.savez_compressed(os.path.join(HERE, name), index=idx, value=g[idx])


def main():
    gold = {}
    with tempfile.TemporaryDirectory() as tmp:
        pre = {}
        for name in DATASETS:
            pre[name] = os.path.join(tmp, name)
            write_dataset(name, pre[name])
            gold[name] = {"bed": sha256(pre[name] + ".bed")}

        # 4,096 x 65,536: KING table under a filter that keeps the top 3 % of the pairs, GRM, LD prune
        d, o = pre["d4k"], os.path.join(tmp, "d4k_ref")
        run(REF, d, ["--make-king", "bin4", "triangle"], o)
        kin = np.fromfile(o + ".king.bin", dtype=np.float32)
        assert kin.size == 4096 * 4095 // 2
        thr = repr(float(np.quantile(kin.astype(np.float64), 0.97)))
        run(REF, d, ["--make-king", "bin4", "triangle", "--make-king-table", "counts", "cols=+ibs1,+ibs", "--king-table-filter", thr], o)
        gold["d4k"]["king_table"] = {"king_table_filter": thr, "kin0_rows": sum(1 for _ in open(o + ".kin0")) - 1,
                                     "king.bin": sha256(o + ".king.bin"), "king.id": sha256(o + ".king.id"), "kin0": sha256(o + ".kin0")}
        run(REF_LAPACK, d, ["--make-grm-bin"], o)
        grm_sample(o, 4096, "scale_d4k_grm_sample.npz")
        gold["d4k"]["grm"] = {"grm.N.bin": sha256(o + ".grm.N.bin"), "grm.id": sha256(o + ".grm.id")}
        run(REF, d, ["--indep-pairwise", "500", "50", "0.2"], o)
        gold["d4k"]["prune"] = {"kept": sum(1 for _ in open(o + ".prune.in")), "prune.in": sha256(o + ".prune.in"), "prune.out": sha256(o + ".prune.out")}

        # 20,000 x 2,048: the whole kinship triangle
        o = os.path.join(tmp, "d20k_ref")
        run(REF, pre["d20k"], ["--make-king", "bin4", "triangle"], o)
        gold["d20k"]["king.bin"] = sha256(o + ".king.bin")

        # 3,000 x 4,096: fp64 matrix and a table that keeps every pair above -0.05
        o = os.path.join(tmp, "d3k_ref")
        run(REF, pre["d3k"], ["--make-king", "bin", "triangle", "--make-king-table", "counts", "--king-table-filter", "-0.05"], o)
        gold["d3k"]["king.bin"], gold["d3k"]["kin0"] = sha256(o + ".king.bin"), sha256(o + ".kin0")

        # 3,000 x 20,000 (two-GPU tests)
        d, o = pre["mg"], os.path.join(tmp, "mg_ref")
        run(REF, d, ["--make-king", "bin", "triangle", "--make-king-table", "counts", "--king-table-filter", "-0.03"], o)
        gold["mg"]["king"] = {ext: sha256(o + "." + ext) for ext in ("king.bin", "kin0", "king.id")}
        run(REF_LAPACK, d, ["--make-grm-bin"], o)
        grm_sample(o, 3000, "scale_mg_grm_sample.npz")
        gold["mg"]["grm.N.bin"] = sha256(o + ".grm.N.bin")

    with open(os.path.join(HERE, "scale_ref.json"), "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
