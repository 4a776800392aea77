"""GPU: parity AT SCALE, through the product (the plink2_b200 host program), against the UNMODIFIED reference
binary.  The inputs are regenerated from a seed (the LD generator of test_ld_gpu.py, written as .bed); what the
reference wrote for the same files is kept in tests/golden/scale_ref.json (SHA-256 digests of the files that must
match byte for byte, row counts, the table filter) and tests/golden/scale_*_grm_sample.npz (a fixed sample of the
GRM entries that are compared within a tolerance); tests/golden/make_scale_set.py regenerates both from
oracle/_ref/plink2[_lapack].

Sizes are the ones SURVEY.md 8(c) names for the smoke set: 4,096 samples x 65,536 variants (32 row tiles x
up to 52 column tiles, two 32,768-variant batches for GRM / several for KING), plus a 20,000-sample KING
run (157 row tiles) that pins tile placement and orientation pair by pair, and a forced multipass run.
"""
import hashlib
import json
import os
import re
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "plink_ng_b200", "plink2_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden")
ENV = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])

# name -> (samples, variants, seed)
DATASETS = {"d4k": (4096, 65536, 1), "d20k": (20000, 2048, 5), "d3k": (3000, 4096, 9), "mg": (3000, 20000, 11)}


def _write_bed(prefix, geno):
    """geno [variants, samples] codes 0/1/2/3 (ALT count, 3 = missing) -> .bed (SNP-major) / .bim / .fam."""
    m, n = geno.shape
    bed_code = np.array([3, 2, 0, 1], dtype=np.uint8)[geno]  # .bed: 00 hom A1(=ALT), 01 missing, 10 het, 11 hom A2(=REF)
    pad = (-n) % 4
    b = np.pad(bed_code, ((0, 0), (0, pad))).reshape(m, -1, 4)
    packed = (b[:, :, 0] | (b[:, :, 1] << 2) | (b[:, :, 2] << 4) | (b[:, :, 3] << 6)).astype(np.uint8)
    with open(prefix + ".bed", "wb") as f:
        f.write(bytes([0x6C, 0x1B, 0x01]))
        packed.tofile(f)
    with open(prefix + ".bim", "w") as f:
        f.write("".join(f"1\tsnp{k}\t0\t{k + 1}\tA\tG\n" for k in range(m)))
    with open(prefix + ".fam", "w") as f:
        f.write("".join(f"0\tper{k}\t0\t0\t2\t-9\n" for k in range(n)))


def write_dataset(name, prefix):
    from test_ld_gpu import _ld_geno

    n, m, seed = DATASETS[name]
    _write_bed(prefix, _ld_geno(m, n, seed=seed))


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def gold(name):
    with open(os.path.join(GOLDEN, "scale_ref.json")) as f:
        return json.load(f)[name]


def dataset(tmp_dir, name):
    """The seeded input fileset; its .bed must be the one the reference results were computed on."""
    pre = str(tmp_dir / name)
    write_dataset(name, pre)
    assert sha256(pre + ".bed") == gold(name)["bed"], f"{name}: the generator no longer writes the input the reference results belong to"
    return pre


def sh(cmd, env=None, ok=(0,)):
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    assert r.returncode in ok, " ".join(cmd) + "\n" + r.stdout[-2000:] + r.stderr[-2000:]
    return r


def assert_same(got, digest, what):
    assert sha256(got) == digest, f"{got} differs from the reference's {what}"


def assert_grm_matches_sample(path, n, sample):
    """fp32 .grm.bin entries at the stored positions within 1e-5 relative of the reference's (LAPACK build, fp64 dsyrk)."""
    got = np.fromfile(path, dtype=np.float32)
    assert got.size == n * (n + 1) // 2
    with np.load(os.path.join(GOLDEN, sample)) as z:
        idx, want = z["index"].astype(np.int64), z["value"].astype(np.float64)
    # fp32 payload: half an ulp of the stored value (6e-8 relative) on top of the 1e-5 relative contract
    b = got[idx].astype(np.float64)
    assert np.allclose(b, want, rtol=1e-5, atol=2e-8), float(np.max(np.abs(want - b)))


@pytest.fixture(scope="module")
def dummy4k(tmp_path_factory):
    return dataset(tmp_path_factory.mktemp("scale4k"), "d4k")


def test_king_table_and_matrix_4096x65536_byte_identical(dummy4k, tmp_path):
    """Every .kin0 count column (NSNP HETHET IBS0 HET1_HOM2 HET2_HOM1 IBS KINSHIP) on a NON-EMPTY filtered table
    (>= 1e5 rows, the top 3 % of the reference's kinship values) plus the whole fp32 kinship triangle, byte for byte."""
    want = gold("d4k")["king_table"]
    out = str(tmp_path / "b200")
    flags = ["--make-king-table", "counts", "cols=+ibs1,+ibs", "--king-table-filter", want["king_table_filter"]]
    sh([BIN, "--bfile", dummy4k] + flags + ["--make-king", "bin4", "triangle", "--out", out], env=ENV)
    rows = sum(1 for _ in open(out + ".kin0")) - 1
    assert rows == want["kin0_rows"] >= 100_000, rows
    assert os.path.getsize(out + ".king.bin") == 4 * (4096 * 4095 // 2)
    assert_same(out + ".king.bin", want["king.bin"], ".king.bin")
    assert_same(out + ".king.id", want["king.id"], ".king.id")
    assert_same(out + ".kin0", want["kin0"], ".kin0")


def test_king_matrix_20000_samples_pairwise(tmp_path):
    """157 row tiles x up to 250 column tiles: the whole 2e8-pair fp32 kinship triangle against the reference's, so a
    tile-placement or orientation error anywhere in the triangle fails (the marginal-sum test cannot see those)."""
    pre, out = dataset(tmp_path, "d20k"), str(tmp_path / "b200")
    sh([BIN, "--bfile", pre, "--make-king", "bin4", "triangle", "--out", out], env=ENV)
    assert os.path.getsize(out + ".king.bin") == 4 * (20000 * 19999 // 2)
    assert_same(out + ".king.bin", gold("d20k")["king.bin"], ".king.bin")


def test_king_forced_multipass_matches_single_pass(tmp_path):
    """--gpu-memory caps the device budget so RunKing needs >= 3 row-block passes (the reference's
    CountTrianglePasses behaviour, 2.0/plink2_matrix_calc.cc:216-255); outputs must not change."""
    pre, one = dataset(tmp_path, "d3k"), str(tmp_path / "one")
    want = gold("d3k")
    flags = ["--make-king", "bin", "triangle", "--make-king-table", "counts", "--king-table-filter", "-0.05"]
    sh([BIN, "--bfile", pre] + flags + ["--out", one], env=ENV)
    assert_same(one + ".king.bin", want["king.bin"], ".king.bin")
    assert_same(one + ".kin0", want["kin0"], ".kin0")
    passes = 0
    for mib in (640, 560, 500, 470, 450, 435, 425, 415):
        multi = str(tmp_path / f"multi{mib}")
        r = sh([BIN, "--bfile", pre] + flags + ["--gpu-memory", str(mib), "--out", multi], env=ENV, ok=(0, 2))
        if r.returncode:
            break  # below the fixed staging buffers: nothing smaller can work
        m = re.search(r"(\d+) passes over the variants", r.stdout)
        passes = int(m.group(1)) if m else 1
        assert_same(multi + ".king.bin", want["king.bin"], f".king.bin (--gpu-memory {mib})")
        assert_same(multi + ".kin0", want["kin0"], f".kin0 (--gpu-memory {mib})")
        if passes >= 3:
            break
    assert passes >= 3, f"no --gpu-memory value produced >= 3 passes (last: {passes})"


def test_grm_4096x65536_vs_reference_blas(dummy4k, tmp_path):
    """.grm.bin against the LAPACK build of the reference (threaded OpenBLAS dsyrk in fp64) within 1e-5 relative on
    every diagonal entry and 4,096 fixed off-diagonal ones (a misplaced 128 x 128 tile is hit with probability
    0.9997), .grm.N.bin (per-pair observation counts) and .grm.id
    exactly."""
    want = gold("d4k")["grm"]
    out = str(tmp_path / "b200")
    sh([BIN, "--bfile", dummy4k, "--make-grm-bin", "--out", out], env=ENV)
    assert_grm_matches_sample(out + ".grm.bin", 4096, "scale_d4k_grm_sample.npz")
    assert_same(out + ".grm.N.bin", want["grm.N.bin"], ".grm.N.bin")
    assert_same(out + ".grm.id", want["grm.id"], ".grm.id")


def test_indep_pairwise_500_50_02_keep_list_4096x65536(dummy4k, tmp_path):
    """The BASELINE config-4 command on the 65,536-variant set: .prune.in / .prune.out byte-identical."""
    want = gold("d4k")["prune"]
    out = str(tmp_path / "b200")
    sh([BIN, "--bfile", dummy4k, "--indep-pairwise", "500", "50", "0.2", "--out", out], env=ENV)
    kept = sum(1 for _ in open(out + ".prune.in"))
    assert 10_000 < want["kept"] < 60_000 and kept == want["kept"], kept
    assert_same(out + ".prune.in", want["prune.in"], ".prune.in")
    assert_same(out + ".prune.out", want["prune.out"], ".prune.out")
