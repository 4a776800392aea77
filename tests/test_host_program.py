"""CPU: host-side pieces of plink2_b200 that need no GPU - the pgenlib reader surface (all three
storage modes incl. difflist / LD-compressed records) and byte-identical number formatting."""
import gzip
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

from oracle import plink_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "plink_ng_b200", "plink2_b200")


def _dump(pgen, psam, pvar, tmp_path):
    out = tmp_path / "geno.bin"
    r = subprocess.run([BIN, "--debug-dump-geno", pgen, psam, pvar, str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return np.fromfile(out, dtype=np.uint8)


@pytest.mark.parametrize("pgen,psam,pvar", [("a.bed", "a.fam", "a.bim"), ("a_mode02.pgen", "a.psam", "a.pvar"), ("a_mode10.pgen", "a.psam", "a.pvar")])
def test_reader_decodes_all_storage_modes(golden_dir, tmp_path, pgen, psam, pvar):
    want = orc.read_bed(os.path.join(golden_dir, "a.bed"), 100)
    got = _dump(os.path.join(golden_dir, pgen), os.path.join(golden_dir, psam), os.path.join(golden_dir, pvar), tmp_path)
    assert np.array_equal(got.reshape(want.shape), want)


def test_reader_on_structure_rich_fixture(golden_dir, tmp_path):
    """Set B (37 samples - not a multiple of 4 -, 400 variants): rare-ALT and rare-REF variants (difflists on either
    base), monomorphic and all-missing variants, 40 % missingness, near-copies of the previous variant
    (LD-compressed records), written by the reference's --make-pgen: our reader must reproduce the .bed exactly,
    full and through a founder-style sample subset."""
    want = orc.read_bed(os.path.join(golden_dir, "b.bed"), 37)
    assert want.shape == (400, 37)
    for pgen, psam, pvar in (("b.bed", "b.fam", "b.bim"), ("b_mode10.pgen", "b.psam", "b.pvar")):
        got = _dump(os.path.join(golden_dir, pgen), os.path.join(golden_dir, psam), os.path.join(golden_dir, pvar), tmp_path)
        assert np.array_equal(got.reshape(400, 37), want), pgen
    # the compressed file really exercises the non-trivial record types
    raw = open(os.path.join(golden_dir, "b_mode10.pgen"), "rb").read()
    assert raw[2] == 0x10 and len(raw) < 0.6 * (3 + 400 * 10)


def test_mode10_fixture_really_uses_compressed_records(golden_dir):
    raw = open(os.path.join(golden_dir, "a_mode10.pgen"), "rb").read()
    assert raw[:3] == b"\x6c\x1b\x10"
    assert len(raw) < 25012  # smaller than the fixed-width file => difflist / LD records present


def test_dtoa_g_matches_reference_text(golden_dir, tmp_path):
    # KINSHIP column of the reference's .kin0 and every entry of its square .king matrix
    geno = orc.read_bed(os.path.join(golden_dir, "a.bed"), 100)
    kin = orc.king_kinship(orc.king_counts(geno))
    extra = np.array([0.0, 1.0, -1.0, 0.5, 123456.7, 1234567.0, 9.9999949e-5, 1e-5, 3.25e-7, 1e300, -2.5e-300, np.inf, -np.inf, np.nan, 0.1, 0.01, 0.001, 0.0001, 99999.95, 999999.5, 0.9999995, 2.0 / 3, 1e15, 1e16])
    vals = np.concatenate([kin, extra])
    fin, fout = tmp_path / "d.bin", tmp_path / "d.txt"
    vals.astype("<f8").tofile(fin)
    r = subprocess.run([BIN, "--debug-dtoa", str(fin), str(fout)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(fout).read().split("\n")[:-1]
    ref_rows = [ln.split("\t") for ln in gzip.open(os.path.join(golden_dir, "a_king.kin0.gz"), "rt").read().split("\n")[1:-1]]
    assert [row[-1] for row in ref_rows] == got[: len(kin)]
    # spot checks against C's %g (same 6-significant-digit contract away from exact ties)
    for x, s in zip(extra, got[len(kin):]):
        if np.isnan(x):
            assert s == "nan"
        elif np.isinf(x):
            assert s == ("inf" if x > 0 else "-inf")
        else:
            assert float(s) == pytest.approx(x, rel=6e-6, abs=0), (x, s)
    assert got[len(kin)] == "0" and got[len(kin) + 3] == "0.5" and got[len(kin) + 7] == "1e-05"


SFMT_DRAWS = 5000


def dtoa_p8_inputs():
    """85,030 doubles: all magnitude ranges, exact .5 ties at every digit position and values a few 1e-7 either side
    of them, zeros, infinities, NaN."""
    rng = np.random.default_rng(5)
    fixed = [0.0, -0.0, 1.0, -1.0, 0.5, 0.1, 0.01, 0.001, 0.0001, 1e-5, 123456.789, 12345678.9, 99999999.4, 99999999.5, 1e8, 1.5e8, 9.9999999e-5, 2 / 3, 1 / 3, np.pi, 1e300,
             -2.5e-300, np.inf, -np.inf, np.nan, 0.99999999, 0.999999995, 0.05, 0.025, 0.0125]
    rnd = np.concatenate([
        rng.uniform(-1, 1, 20000), 10 ** rng.uniform(-12, 12, 20000) * rng.choice([-1, 1], 20000), rng.uniform(0, 0.2, 20000),
        (rng.integers(1, 10 ** 8, 20000) + 0.5) / 10.0 ** rng.integers(0, 9, 20000),
        (rng.integers(1, 10 ** 8, 5000) + 0.5 + rng.choice([-1e-7, 1e-7, 3e-7, -3e-7], 5000)) / 10.0 ** rng.integers(0, 9, 5000)])
    return np.concatenate([np.array(fixed), rnd]).astype("<f8")


def test_dtoa_g_p8_matches_reference_function(golden_dir, tmp_path):
    """The 8-digit formatter behind --make-grm-sparse, byte for byte against the reference's own dtoa_g_p8
    (2.0/include/plink2_string.cc:2641) on dtoa_p8_inputs(); tests/golden/dtoa_g_p8.json holds the digest of the
    reference's text (make_host_format_set.py)."""
    vals = dtoa_p8_inputs()
    vals.tofile(tmp_path / "in.bin")
    subprocess.run([BIN, "--debug-dtoa-p8", str(tmp_path / "in.bin"), str(tmp_path / "got.txt")], check=True)
    want = json.load(open(os.path.join(golden_dir, "dtoa_g_p8.json")))
    raw = open(tmp_path / "got.txt", "rb").read()
    got = raw.decode().split("\n")
    assert want["lines"] == len(vals) and len(got) == len(vals) + 1
    assert got[10] == "123456.79" and got[17] == "0.66666667" and got[22] == " inf"
    assert hashlib.sha256(raw).hexdigest() == want["sha256"]


def test_sfmt_and_gaussian_fill_match_reference_generator(golden_dir, tmp_path):
    """The SFMT-19937 restatement and FillGaussian reproduce the reference's vendored generator
    (2.0/include/SFMT.c; its first draws for seed 11 are tests/golden/sfmt_seed11.u32, make_host_format_set.py) and
    RandNormal/FillGaussianDArr (2.0/plink2_random.cc:29-99) bit for bit."""
    n = SFMT_DRAWS
    subprocess.run([BIN, "--debug-sfmt", "11", str(n), str(tmp_path / "got.u32")], check=True)
    ref = np.fromfile(os.path.join(golden_dir, "sfmt_seed11.u32"), dtype="<u4")
    got = np.fromfile(tmp_path / "got.u32", dtype=np.uint32)
    assert ref.size == n and np.array_equal(ref, got)
    # Gaussian fill, single stream: Box-Muller on consecutive draws
    subprocess.run([BIN, "--debug-gauss", "11", "1000", "1", str(tmp_path / "g.f64")], check=True)
    g = np.fromfile(tmp_path / "g.f64", dtype=np.float64)
    u = (ref[:2000].astype(np.float64) + 0.5) * 2.0 ** -32
    r = np.sqrt(-2 * np.log(u[0::2]))
    th = (2 * 3.1415926535897932) * u[1::2]
    assert np.allclose(g[0::2], r * np.sin(th), rtol=1e-15, atol=0) and np.allclose(g[1::2], r * np.cos(th), rtol=1e-15, atol=0)
    # two streams (pairs > 262144): the second half comes from an init_by_array-seeded generator
    pairs = 300000
    subprocess.run([BIN, "--debug-gauss", "11", str(pairs), "4", str(tmp_path / "g2.f64")], check=True)
    g2 = np.fromfile(tmp_path / "g2.f64", dtype=np.float64)
    assert g2.shape[0] == 2 * pairs and np.isfinite(g2).all() and abs(g2.mean()) < 0.01 and abs(g2.std() - 1) < 0.01


@pytest.mark.parametrize("flags,fragment", [
    (("--glm",), "unsupported"),
    (("--make-grm-bin", "--make-grm-list"), "--make-grm-list cannot be used with --make-grm-bin"),
    (("--score", "w.txt", "se"), "not supported"),
    (("--indep-preferred", "x.txt"), "--indep-preferred must be used with --indep-pairwise"),
    (("--make-king-table", "--king-table-subset"), "--king-table-subset requires"),
    (("--pca", "0"), "Invalid --pca PC count"),
    (("--indep-pairwise", "50"), "--indep-pairwise requires 2-4 arguments"),
    (("--make-grm-sparse", "0.05", "--make-grm-bin"), "cannot be used with --make-grm-sparse"),
    (("--make-grm-sparse", "abc"), "Invalid --make-grm-sparse threshold"),
])
def test_command_line_errors_exit_8_before_touching_the_gpu(golden_dir, tmp_path, flags, fragment):
    """kPglRetInvalidCmdline = 8, as the reference; the command line is validated before any CUDA call, so this
    runs on a machine without a GPU."""
    r = subprocess.run([BIN, "--bfile", os.path.join(golden_dir, "a"), *flags, "--out", str(tmp_path / "x")], capture_output=True, text=True)
    assert r.returncode == 8, r.stdout + r.stderr
    assert fragment in r.stdout + r.stderr


def test_no_gpu_means_loud_failure_not_a_cpu_fallback(golden_dir, tmp_path):
    """Without a visible device the program must stop with kPglRetGpuFail-style code 16 - there is no CPU path."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([BIN, "--bfile", os.path.join(golden_dir, "a"), "--make-king-table", "--out", str(tmp_path / "x")], capture_output=True, text=True, env=env)
    assert r.returncode == 16, r.stdout + r.stderr
    assert "GPU" in r.stdout
    assert not os.path.exists(str(tmp_path / "x") + ".kin0")


def test_zs_writer_roundtrip(tmp_path):
    """OutFile's Zstandard mode (the 'zs' output modifiers): frames written through libzstd decompress to the input."""
    import ctypes as C

    import numpy as np

    data = np.random.default_rng(0).integers(0, 7, size=5_000_000, dtype=np.uint8).tobytes()
    (tmp_path / "in.bin").write_bytes(data)
    subprocess.run([BIN, "--debug-zst", str(tmp_path / "in.bin"), str(tmp_path / "out.zst")], check=True)
    raw = (tmp_path / "out.zst").read_bytes()
    assert len(raw) < len(data) // 2
    z = C.CDLL("libzstd.so.1")
    z.ZSTD_findFrameCompressedSize.restype = C.c_size_t
    z.ZSTD_findFrameCompressedSize.argtypes = [C.c_void_p, C.c_size_t]
    z.ZSTD_getFrameContentSize.restype = C.c_ulonglong
    z.ZSTD_getFrameContentSize.argtypes = [C.c_void_p, C.c_size_t]
    z.ZSTD_decompress.restype = C.c_size_t
    z.ZSTD_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    buf = C.create_string_buffer(raw, len(raw))
    base, off, out = C.addressof(buf), 0, b""
    while off < len(raw):
        fsz = z.ZSTD_findFrameCompressedSize(base + off, len(raw) - off)
        n = z.ZSTD_getFrameContentSize(base + off, fsz)
        dst = C.create_string_buffer(int(n))
        assert z.ZSTD_decompress(dst, n, base + off, fsz) == n
        out += dst.raw[:n]
        off += fsz
    assert out == data


def test_king_cutoff_table_matches_reference_lists(tmp_path):
    """--king-cutoff-table is host-only work in the reference as well (KingCutoffBatchTable): the .kin0 table the
    reference wrote for set A, threshold 0.02 -> the reference's .king.cutoff.{in,out}.id, byte for byte, no GPU needed."""
    import gzip

    gd = os.path.join(ROOT, "tests", "golden")
    (tmp_path / "in.kin0").write_bytes(gzip.open(os.path.join(gd, "a_kingp.kin0.gz"), "rb").read())
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--bfile", os.path.join(gd, "a"), "--king-cutoff-table", str(tmp_path / "in.kin0"), "0.02", "--out", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "661 constraints loaded" in r.stdout
    for ext in (".king.cutoff.in.id", ".king.cutoff.out.id"):
        assert open(out + ext, "rb").read() == open(os.path.join(gd, "a_kct" + ext), "rb").read()
    # set R has real FIDs.  A table without FID columns reads its IDs with FID 0 (XidRead, plink2_common.cc:1280), so it
    # names nobody there: the reference loads 0 constraints from the first table and 1 from the second (checked here).
    (tmp_path / "iid.kin0").write_text("#IID1\tIID2\tKINSHIP\n9\tp\t0.4\n")
    (tmp_path / "fid.kin0").write_text("#FID1\tIID1\tFID2\tIID2\tKINSHIP\nF1\t9\tF1\tp\t0.4\n")
    for name, want in (("iid.kin0", "0 constraints loaded"), ("fid.kin0", "1 constraint loaded")):
        r = subprocess.run([BIN, "--bfile", os.path.join(gd, "r"), "--king-cutoff-table", str(tmp_path / name), "0.1", "--out", out], capture_output=True, text=True)
        assert r.returncode == 0 and want in r.stdout, r.stdout + r.stderr


def test_king_cutoff_matrix_prefix_matches_reference_lists(tmp_path):
    """`--king-cutoff <prefix> <threshold>` (KingCutoffBatchBinary, 2.0/plink2_matrix_calc.cc:393): (1) the reference's
    fp32 triangle over set A - 661 constraints against the threshold rounded to fp32, where the fp64 matrix gives 662;
    (2) an fp64 triangle over a shuffled 80-ID subset whose ID file also lists three unknown samples.  Host-only work:
    lists byte-identical to the reference's, no GPU needed.  A square matrix and an IID-only ID file on a FID-bearing
    dataset fail the way the reference does."""
    import shutil

    gd = os.path.join(ROOT, "tests", "golden")
    shutil.copy(os.path.join(gd, "a_king.king.bin"), tmp_path / "kc4.king.bin")
    shutil.copy(os.path.join(gd, "a_kingsq.king.id"), tmp_path / "kc4.king.id")
    for prefix, thr, want, gold in ((str(tmp_path / "kc4"), "0.02", "661 constraints", "a_kc4"), (os.path.join(gd, "a_kc8"), "0.03", "250 constraints", "a_kc8")):
        out = str(tmp_path / ("o_" + gold))
        r = subprocess.run([BIN, "--bfile", os.path.join(gd, "a"), "--king-cutoff", prefix, thr, "--out", out], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        assert want + " loaded" in r.stdout
        for ext in (".king.cutoff.in.id", ".king.cutoff.out.id"):
            assert open(out + ext, "rb").read() == open(os.path.join(gd, gold + ext), "rb").read()
    # square matrix: refused
    n = 100
    (tmp_path / "sq.king.bin").write_bytes(b"\0" * (4 * n * n))
    shutil.copy(os.path.join(gd, "a_kingsq.king.id"), tmp_path / "sq.king.id")
    r = subprocess.run([BIN, "--bfile", os.path.join(gd, "a"), "--king-cutoff", str(tmp_path / "sq"), "0.1", "--out", str(tmp_path / "x")], capture_output=True, text=True)
    assert r.returncode != 0 and "appears to be square" in r.stdout + r.stderr
    # set R carries real FIDs: an ID file without a FID column reads every ID with FID 0 and matches nothing
    fam = [l.split() for l in open(os.path.join(gd, "r.fam"))]
    (tmp_path / "r.king.id").write_text("#IID\n" + "".join(f[1] + "\n" for f in fam))
    (tmp_path / "r.king.bin").write_bytes(b"\0" * (4 * len(fam) * (len(fam) - 1) // 2))
    r = subprocess.run([BIN, "--bfile", os.path.join(gd, "r"), "--king-cutoff", str(tmp_path / "r"), "0.1", "--out", str(tmp_path / "x")], capture_output=True, text=True)
    assert r.returncode != 0 and "expected 0 or 0 bytes" in r.stdout + r.stderr


FILTER_CASES = [
    # (dataset arguments, filter arguments, golden prefix, extensions compared)
    (["--bfile", "x"], ["--keep", "x_keep1.txt", "x_keep2.txt", "--remove", "x_remove.txt", "--extract", "x_extract.txt", "--exclude", "x_exclude.txt"], "x_filt", ("bed", "bim", "fam")),
    (["--bfile", "x"], ["--chr", "1,X,Y", "--not-chr", "Y"], "x_chr", ("bed", "bim")),
    (["--pgen", "a_mode10.pgen", "--pvar", "a.pvar", "--psam", "a.psam"], ["--remove", "x_remove.txt", "--exclude", "x_exclude.txt"], "a_filt", ("bed", "bim", "fam")),
    (["--bfile", "s"], ["--keep-fam", "s_keepfam.txt", "--remove-fam", "s_removefam.txt"], "s_famfilt", ("bed", "fam")),
]


@pytest.mark.parametrize("case", range(len(FILTER_CASES)))
def test_filters_and_make_bed_match_reference(tmp_path, case):
    """The sample / variant filters in front of every command (--keep, --remove, --keep-fam, --remove-fam, --extract,
    --exclude, --chr, --not-chr) compact the dataset and install a view in the genotype reader; --make-bed writes that
    view.  Host-only, so checked here: .bed / .bim / .fam byte-identical to the reference's --make-bed under the same
    filters, for a .bed input with sex chromosomes, an LD-compressed .pgen, and FID-based lists."""
    gd = os.path.join(ROOT, "tests", "golden")
    data, filt, gold, exts = FILTER_CASES[case]
    out = str(tmp_path / "o")
    r = subprocess.run([BIN] + data + filt + ["--make-bed", "--threads", "3", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in exts:
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, gold + "." + ext), "rb").read(), ext
    if case == 0:
        assert "--keep: 80 samples remaining." in r.stdout and "--remove: 60 samples remaining." in r.stdout
        assert "--extract: 500 variants remaining." in r.stdout and "--exclude: 420 variants remaining." in r.stdout
        assert "duplicate ID in --keep" in r.stdout


QC_CASES = [
    (["--bfile", "x"], ["--keep", "x_keep1.txt", "x_keep2.txt", "--mind", "0.035", "--geno", "0.02", "--maf", "0.05"], "x_qc", ("bed", "bim", "fam", "mindrem.id")),
    (["--bfile", "x"], ["--keep-founders", "--mac", "30", "--max-maf", "0.45"], "x_mac", ("bim", "fam")),
    (["--bfile", "x"], ["--remove-nosex", "--keep-nonfounders"], "x_sex", ("fam",)),
    (["--pgen", "a_mode10.pgen", "--pvar", "a.pvar", "--psam", "a.psam"], ["--geno", "0.03", "--mind", "0.04", "--maf", "0.2"], "a_qc", ("bed", "bim", "fam")),
    (["--bfile", "a"], ["--read-freq", "a_rf.afreq", "--exclude", "x_exclude.txt", "--maf", "0.3"], "a_rfmaf", ("bim",)),  # thresholds on LOADED frequencies
    (["--bfile", "x"], ["--nonfounders", "--maf", "0.1", "--mac", "30"], "x_nf", ("bim",)),  # frequencies / allele counts over all samples
    (["--bfile", "x"], ["--bp-space", "7", "--maf", "0.05", "--chr", "1,X,MT"], "x_bpspace", ("bim",)),  # spacing filter applied after the frequency thresholds
]


@pytest.mark.parametrize("case", range(len(QC_CASES)))
def test_count_based_filters_match_reference(tmp_path, case):
    """--mind, --geno, --maf / --max-maf / --mac and the sex / founder filters: one host counting pass over the view
    (chrY missingness over males only, founder frequencies with the chrX / chrY / MT allele accounting of --freq),
    thresholds with the reference's 2^-44 guard.  Same survivors as the reference, byte for byte, through --make-bed."""
    gd = os.path.join(ROOT, "tests", "golden")
    data, filt, gold, exts = QC_CASES[case]
    out = str(tmp_path / "o")
    r = subprocess.run([BIN] + data + filt + ["--make-bed", "--threads", "3", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in exts:
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, gold + "." + ext), "rb").read(), ext
    if case == 0:
        assert "27 samples removed due to missing genotype data (--mind)." in r.stdout
        assert "--geno: 283 variants removed" in r.stdout and "65 variants removed due to allele frequency threshold(s)" in r.stdout
    if case == 1:
        # nonfounders present: the reference refuses allele-count thresholds without --ac-founders / --nonfounders
        r = subprocess.run([BIN] + data + ["--mac", "30", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
        assert r.returncode == 7 and "nonfounders are present" in r.stdout


def test_allele_and_position_filters_and_id_lists(tmp_path):
    """--snps-only [just-acgt] on a .bim with indels, symbolic alleles, lower case and both missing-allele codes (a lone
    '0' is stored and written as '.'), --chr + --from-kb/--to-kb (lower bound rounded up, upper bound down), and the
    --write-snplist / --write-samples lists of what the filters left - all as the reference writes them."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    for mod, gold in (([], "x_snps.bim"), (["just-acgt"], "x_acgt.bim")):
        r = subprocess.run([BIN, "--bed", "x.bed", "--bim", "x_alleles.bim", "--fam", "x.fam", "--snps-only"] + mod + ["--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
        assert r.returncode == 0, r.stdout + r.stderr
        assert open(out + ".bim", "rb").read() == open(os.path.join(gd, gold), "rb").read(), gold
    r = subprocess.run([BIN, "--bfile", "x", "--chr", "1", "--from-kb", "0.1001", "--to-kb", "0.25", "--keep", "x_keep2.txt", "--write-snplist", "--write-samples", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    assert open(out + ".snplist", "rb").read() == open(os.path.join(gd, "x_bp.snplist"), "rb").read()
    assert open(out + ".id", "rb").read() == open(os.path.join(gd, "x_bp.id"), "rb").read()
    r = subprocess.run([BIN, "--bfile", "x", "--chr", "1,2", "--from-bp", "5", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode != 0 and "only one chromosome" in r.stdout + r.stderr


def test_compressed_text_inputs(tmp_path):
    """Every text input goes through one reader that recognises Zstandard and gzip (incl. multi-member / bgzf) by magic
    number, like the reference's TextStream: a .pvar.zst written by the reference, gzipped ID lists (one of them two
    concatenated members), the gzipped golden .kin0 as a --king-cutoff-table input, and a .zst written by this program's
    own 'zs' writer fed back in."""
    import gzip

    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--bed", "x.bed", "--pvar", "x.pvar.zst", "--fam", "x.fam", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    assert open(out + ".bim", "rb").read() == open(os.path.join(gd, "x.bim"), "rb").read()
    assert open(out + ".bed", "rb").read() == open(os.path.join(gd, "x.bed"), "rb").read()
    k1 = open(os.path.join(gd, "x_keep1.txt"), "rb").read().split(b"\n")
    (tmp_path / "k1.gz").write_bytes(gzip.compress(b"\n".join(k1[:5]) + b"\n") + gzip.compress(b"\n".join(k1[5:])))
    (tmp_path / "k2.gz").write_bytes(gzip.compress(open(os.path.join(gd, "x_keep2.txt"), "rb").read()))
    r = subprocess.run([BIN, "--bfile", "x", "--keep", str(tmp_path / "k1.gz"), str(tmp_path / "k2.gz"), "--remove", "x_remove.txt", "--extract", "x_extract.txt", "--exclude", "x_exclude.txt", "--make-bed", "--out", out],
                       capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("bed", "bim", "fam"):
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "x_filt." + ext), "rb").read(), ext
    r = subprocess.run([BIN, "--bfile", "a", "--king-cutoff-table", "a_kingp.kin0.gz", "0.02", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0 and "661 constraints loaded" in r.stdout
    (tmp_path / "in.kin0").write_bytes(gzip.open(os.path.join(gd, "a_kingp.kin0.gz"), "rb").read())
    assert subprocess.run([BIN, "--debug-zst", str(tmp_path / "in.kin0"), str(tmp_path / "in.kin0.zst")]).returncode == 0
    r = subprocess.run([BIN, "--bfile", "a", "--king-cutoff-table", str(tmp_path / "in.kin0.zst"), "0.02", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0 and "661 constraints loaded" in r.stdout
    assert open(out + ".king.cutoff.in.id", "rb").read() == open(os.path.join(gd, "a_kct.king.cutoff.in.id"), "rb").read()
    (tmp_path / "bad.zst").write_bytes(open(tmp_path / "in.kin0.zst", "rb").read()[:200])
    r = subprocess.run([BIN, "--bfile", "a", "--king-cutoff-table", str(tmp_path / "bad.zst"), "0.02", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode != 0 and "Zstandard" in r.stdout


def test_ped_map_import_matches_reference(tmp_path):
    """--pedmap / --ped + --map: the legacy text fileset is converted to a temporary binary fileset first (REF = major
    allele, provisional alleles in order of appearance, negative-bp variants dropped, both .ped layouts), then read
    like any other input.  --make-bed of the result is byte-identical to the reference's for set P (multi-character
    alleles, missing calls, comment line, 4-column .map) and its compound-genotypes twin; the temporary files are gone
    afterwards; half-missing and third-allele calls are refused with the reference's messages."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--pedmap", "p", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("bed", "bim", "fam"):
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "p." + ext), "rb").read(), ext
    assert not [f for f in os.listdir(tmp_path) if "temporary" in f]
    r = subprocess.run([BIN, "--ped", "pc.ped", "--map", "pc.map", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("bed", "bim"):
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "pc." + ext), "rb").read(), ext
    (tmp_path / "h.map").write_text("1 v1 0 10\n1 v2 0 20\n")
    (tmp_path / "h.ped").write_text("0 a 0 0 1 1 A A C 0\n")
    r = subprocess.run([BIN, "--pedmap", str(tmp_path / "h"), "--make-bed", "--out", out], capture_output=True, text=True)
    assert r.returncode == 6 and "Half-missing genotype on line 1" in r.stdout
    (tmp_path / "h.ped").write_text("0 a 0 0 1 1 A C G G\n0 b 0 0 1 1 A T G G\n")
    r = subprocess.run([BIN, "--pedmap", str(tmp_path / "h"), "--make-bed", "--out", out], capture_output=True, text=True)
    assert r.returncode == 6 and "Multiallelic variant" in r.stdout
    # BASELINE.json configs[0] is a .ped/.map pair (2 samples x 2 variants, one all-missing call, one unseen ALT): its
    # content, typed in here, must import to the toy.bed/.bim/.fam the reference produced from its own copy
    (tmp_path / "toy.ped").write_text("1 1000000000 0 0 1 1 0 0 A A\n1 1000000001 0 0 1 2 C C A G\n")
    (tmp_path / "toy.map").write_text("1\trs0\t0\t1000\n1\trs10\t0\t1001\n")
    r = subprocess.run([BIN, "--pedmap", str(tmp_path / "toy"), "--make-bed", "--out", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("bed", "bim", "fam"):
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "toy." + ext), "rb").read(), ext


def test_max_alleles_lets_a_file_with_multiallelic_records_through(tmp_path):
    """Real .pgen files carry some multiallelic variants; `--max-alleles 2` (what plink2 users pass) removes them in the
    variant view, so their records are never decoded as data.  One of them IS still read - as the LD base of the
    biallelic record behind it, whose main track has the biallelic layout.  Result byte-identical to the reference's,
    multi-threaded and single-threaded; without the filter the file is refused with a pointer to the flag."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    for threads in ("1", "4"):
        r = subprocess.run([BIN, "--pfile", "ma", "--max-alleles", "2", "--threads", threads, "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "20 variants excluded" in r.stdout
        for ext in ("bed", "bim"):
            assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "ma_bi." + ext), "rb").read(), ext
    r = subprocess.run([BIN, "--pfile", "ma", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode != 0 and "--max-alleles 2" in r.stdout


def test_variant_id_templates(tmp_path):
    """--set-missing-var-ids / --set-all-var-ids (the usual fix for the duplicate '.' IDs that --indep-pairwise refuses):
    '@' chromosome, '#' position, $r / $a / $1 / $2 alleles - a '0' missing-allele code stays '0' inside the ID even
    though the allele itself is stored as '.'.  IDs as the reference assigns them."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--bed", "x.bed", "--bim", "x_noid.bim", "--fam", "x.fam", "--set-missing-var-ids", "@:#:$1:$2", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    assert open(out + ".bim", "rb").read() == open(os.path.join(gd, "x_setid.bim"), "rb").read()
    r = subprocess.run([BIN, "--bfile", "x", "--set-all-var-ids", "@_#", "--chr", "MT", "--write-snplist", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0 and open(out + ".snplist").read().split()[:2] == ["MT_700", "MT_701"]
    r = subprocess.run([BIN, "--bfile", "x", "--set-all-var-ids", "nochrom", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode != 0 and "template must contain" in r.stdout + r.stderr


def test_make_pgen_writes_a_fileset_every_reader_accepts(tmp_path):
    """--make-pgen: fixed-width .pgen (storage mode 0x02) + .pvar + .psam of the filtered view.  The text files are the
    reference's byte for byte (column rules: FID / PAT+MAT / CM / PHENO1 only when informative); the .pgen is read
    back by this program's own reader and must reproduce the .bed the reference wrote for the same view.  The .pgen itself is the one the reference writes for the
    same view in the same storage mode (`--make-pgen format=2`), byte for byte."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--bfile", "x", "--keep", "x_keep1.txt", "x_keep2.txt", "--extract", "x_extract.txt", "--make-pgen", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("pvar", "psam"):
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "x_mp." + ext), "rb").read(), ext
    raw = open(out + ".pgen", "rb").read()
    assert raw[:3] == b"\x6c\x1b\x02" and int.from_bytes(raw[3:7], "little") == 500 and int.from_bytes(raw[7:11], "little") == 80 and raw[11] == 0x80
    back = str(tmp_path / "back")
    r = subprocess.run([BIN, "--pfile", out, "--make-bed", "--out", back], capture_output=True, text=True)
    assert r.returncode == 0 and open(back + ".bed", "rb").read() == open(os.path.join(gd, "x_mp.bed"), "rb").read()
    assert raw == open(os.path.join(gd, "x_mp.pgen"), "rb").read()
    r = subprocess.run([BIN, "--pedmap", "p", "--make-pgen", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("pvar", "psam"):  # CM column (a nonzero centimorgan exists), PAT / MAT columns, NA sex and phenotype
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "p_mp." + ext), "rb").read(), ext


def test_output_chr_styles(tmp_path):
    """--output-chr: 26 / M / MT with or without the chr prefix, for every file that prints a chromosome (here .bim and,
    through the '@' of an ID template, the IDs); extra contigs are left as written.  Spellings as the reference prints
    them for set X (1, X, Y, XY, MT)."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    want = {"26": ["1", "23", "24", "25", "26"], "M": ["1", "X", "Y", "XY", "M"], "chrMT": ["chr1", "chrX", "chrY", "chrXY", "chrMT"], "chr26": ["chr1", "chr23", "chr24", "chr25", "chr26"]}
    for code, names in want.items():
        r = subprocess.run([BIN, "--bfile", "x", "--output-chr", code, "--set-all-var-ids", "@:#", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
        assert r.returncode == 0, r.stdout + r.stderr
        rows = [ln.split("\t") for ln in open(out + ".bim")]
        seen = list(dict.fromkeys(r_[0] for r_ in rows))
        assert seen == names
        assert all(r_[1] == r_[0] + ":" + r_[3] for r_ in rows)
    r = subprocess.run([BIN, "--bed", "x.bed", "--bim", "x_contigs.bim", "--fam", "x.fam", "--allow-extra-chr", "--output-chr", "chrM", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0 and list(dict.fromkeys(ln.split("\t")[0] for ln in open(out + ".bim"))) == ["chr1", "chrX", "chrY", "chrUn_KI270", "GL000.1", "chrM"]
    r = subprocess.run([BIN, "--bfile", "x", "--output-chr", "0M", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode != 0


def test_split_chromosome_is_refused(tmp_path):
    """A chromosome that reappears after another one is an input error in the reference ("has a split chromosome") and
    would silently become two LD-prune units here, so it is refused at load."""
    gd = os.path.join(ROOT, "tests", "golden")
    rows = open(os.path.join(gd, "a.bim")).read().split("\n")
    rows[10] = "2" + rows[10][1:]
    (tmp_path / "split.bim").write_text("\n".join(rows))
    r = subprocess.run([BIN, "--bed", os.path.join(gd, "a.bed"), "--bim", str(tmp_path / "split.bim"), "--fam", os.path.join(gd, "a.fam"), "--make-bed", "--out", str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode != 0 and "split chromosome" in r.stdout


def test_missing_reports(tmp_path):
    """--missing: .smiss / .vmiss as the reference writes them - for the samples the filters (incl. --mind) left, but
    over the variants BEFORE --geno; chrY calls counted for males only; PHENO1 column = phenotype missing Y/N."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--bfile", "x", "--keep", "x_keep1.txt", "x_keep2.txt", "--mind", "0.05", "--geno", "0.05", "--missing", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("smiss", "vmiss"):
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "x_miss." + ext), "rb").read(), ext
    r = subprocess.run([BIN, "--bfile", "x", "--missing", "variant-only", "zs", "--out", out + "2"], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0 and os.path.exists(out + "2.vmiss.zst") and not os.path.exists(out + "2.smiss.zst")


def test_founder_subset_of_a_filtered_view(tmp_path):
    """LD prune and the allele-frequency pass decode only the founders of whatever the filters left: a sample_include
    bitset over the VIEW's samples, composed with the view's own raw-sample bitset inside the reader.  The hidden
    --debug-founders-bed flag writes exactly that decode; the reference's --keep-founders under the same filters gives
    the expected bytes."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    r = subprocess.run([BIN] + FILTER_CASES[0][0] + FILTER_CASES[0][1] + ["--debug-founders-bed", "--threads", "2", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 0, r.stdout + r.stderr
    assert open(out + ".bed", "rb").read() == open(os.path.join(gd, "x_filt_founders.bed"), "rb").read()


def test_make_bed_round_trips_every_input_mode(tmp_path):
    """Without filters --make-bed must reproduce the .bed the fixtures were converted from: .bed input, fixed-width
    .pgen (mode 0x02) and variable-width .pgen with difflist / LD-compressed records (mode 0x10)."""
    gd = os.path.join(ROOT, "tests", "golden")
    for data in (["--bfile", "a"], ["--pgen", "a_mode02.pgen", "--pvar", "a.pvar", "--psam", "a.psam"], ["--pgen", "a_mode10.pgen", "--pvar", "a.pvar", "--psam", "a.psam"], ["--pgen", "b_mode10.pgen", "--pvar", "b.pvar", "--psam", "b.psam"]):
        out = str(tmp_path / "o")
        r = subprocess.run([BIN] + data + ["--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
        assert r.returncode == 0, r.stdout + r.stderr
        want = "b" if data[1].startswith("b") else "a"
        assert open(out + ".bed", "rb").read() == open(os.path.join(gd, want + ".bed"), "rb").read(), data
        assert open(out + ".bim", "rb").read() == open(os.path.join(gd, want + ".bim"), "rb").read(), data


def test_filter_edge_cases(tmp_path):
    """An ID list without a FID column names only FID-0 samples (set S carries real FIDs -> nobody left, the
    reference's error); unknown chromosome codes and reversed ranges are refused at the command line."""
    gd = os.path.join(ROOT, "tests", "golden")
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--bfile", "s", "--keep", "s_keep_iid.txt", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 7 and "--keep: 0 samples remaining." in r.stdout and "No samples remaining after main filters." in r.stdout
    r = subprocess.run([BIN, "--bfile", "x", "--chr", "1,X-Y", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode != 0 and "cannot be the end of a range" in r.stdout + r.stderr
    r = subprocess.run([BIN, "--bfile", "x", "--chr", "5-3", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode != 0 and "is not greater than" in r.stdout + r.stderr
    r = subprocess.run([BIN, "--bfile", "x", "--extract", "no_such_file.txt", "--make-bed", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 3
    # the LD sample-size guard runs on what the main filters left, before any device work (plink2.cc:2065)
    r = subprocess.run([BIN, "--bfile", "x", "--keep", "x_keep2.txt", "--indep-pairwise", "50", "5", "0.2", "--out", out], capture_output=True, text=True, cwd=gd)
    assert r.returncode == 13 and "less than 50 samples" in r.stdout


def test_relatedness_prune_feeds_later_commands(tmp_path):
    """`--king-cutoff-table ... --make-bed`: the samples removed by the prune are gone from the later command's view,
    as in the reference (plink2.cc:2523-2581) - .fam / .bed identical to the reference's chained run."""
    import gzip

    gd = os.path.join(ROOT, "tests", "golden")
    (tmp_path / "in.kin0").write_bytes(gzip.open(os.path.join(gd, "a_kingp.kin0.gz"), "rb").read())
    out = str(tmp_path / "o")
    r = subprocess.run([BIN, "--bfile", os.path.join(gd, "a"), "--king-cutoff-table", str(tmp_path / "in.kin0"), "0.02", "--make-bed", "--out", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    for ext in ("fam", "bed"):
        assert open(out + "." + ext, "rb").read() == open(os.path.join(gd, "a_kctb." + ext), "rb").read(), ext
    assert open(out + ".king.cutoff.in.id", "rb").read() == open(os.path.join(gd, "a_kct.king.cutoff.in.id"), "rb").read()


def test_natural_sort_matches_reference_order(tmp_path):
    """The ID order behind `--make-king-table rel-check`: the reference's own table on set S (300 random IDs of the
    alphabet aAbBzZ0019_.-x over FIDs F1 / F2 / f1 / F10 / F02) lists every FID block in natural order; the host
    program's comparator must put the same keys in the same order."""
    import gzip

    gd = os.path.join(ROOT, "tests", "golden")
    rows = [ln.split("\t") for ln in gzip.open(os.path.join(gd, "s_relcheck.kin0.gz"), "rt").read().split("\n")[1:] if ln]
    order, seen = [], set()
    for r in rows:
        for key in ((r[2], r[3]), (r[0], r[1])):
            if key not in seen:
                seen.add(key)
                order.append(key[0] + "\t" + key[1])
    fam = [ln.split("\t")[:2] for ln in open(os.path.join(gd, "s.fam"))]
    keys = [f + "\t" + i for f, i in fam if f + "\t" + i in set(order)]
    assert len(keys) == len(order) > 250 and keys != order
    (tmp_path / "in.txt").write_text("\n".join(keys) + "\n")
    subprocess.run([BIN, "--debug-natural-sort", str(tmp_path / "in.txt"), str(tmp_path / "out.txt")], check=True)
    assert (tmp_path / "out.txt").read_text().split("\n")[:-1] == order


def test_rel_check_pair_list_matches_reference_table(tmp_path):
    """The pair list behind `--make-king-table rel-check` (natural sort + the reference's FID-block rule, which also joins
    FIDs that differ only in capitalisation): ID columns of the reference's own tables, in order, for both fixtures."""
    import gzip

    gd = os.path.join(ROOT, "tests", "golden")
    for prefix, table in (("r", "r_relcheck.kin0"), ("s", "s_relcheck.kin0.gz")):
        path = os.path.join(gd, table)
        text = gzip.open(path, "rt").read() if table.endswith(".gz") else open(path).read()
        want = ["\t".join(ln.split("\t")[:4]) for ln in text.split("\n")[1:] if ln]
        subprocess.run([BIN, "--debug-rel-check-pairs", os.path.join(gd, prefix + ".fam"), str(tmp_path / "p.txt")], check=True)
        assert (tmp_path / "p.txt").read_text().split("\n")[:-1] == want, prefix


def test_read_freq_parser_counts_match_the_reference_log(tmp_path):
    """--read-freq parsing happens before any device is touched: the counts the reference logs for the same file
    ("Frequencies for 849 variants loaded", "60 entries skipped") must come out on a box without a GPU too (the run then
    stops with exit code 16 at GPU initialisation, or completes when a device is present)."""
    gd = os.path.join(ROOT, "tests", "golden")
    r = subprocess.run([BIN, "--bfile", os.path.join(gd, "a"), "--read-freq", os.path.join(gd, "a_rf.afreq"), "--make-grm-bin", "--out", str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode in (0, 16), r.stdout + r.stderr
    assert "--read-freq: PLINK 2 --freq file detected." in r.stdout
    assert "--read-freq: Frequencies for 849 variants loaded." in r.stdout
    assert "Warning: 60 entries skipped" in r.stdout


def test_view_and_subset_decode_against_a_numpy_model(tmp_path):
    """Property test of the reader view: random --keep lists (so the raw-sample keep bitset has arbitrary gaps across
    the 32- and 64-sample word boundaries) composed with a random founder subset of the view (the sample_include a
    founder-only command passes), on set S's genotypes (300 samples = five 64-sample words) under a .fam with about half the samples marked as non-founders.
    The .bed the program writes for "founders of the kept samples" must equal the same selection done with numpy."""
    gd = os.path.join(ROOT, "tests", "golden")
    rng = np.random.default_rng(2026)
    fam = [ln.split() for ln in open(os.path.join(gd, "s.fam"))]
    n = len(fam)
    geno = orc.read_bed(os.path.join(gd, "s.bed"), n)  # [variants, samples], codes 0..3
    to_bed = np.array([3, 2, 0, 1], dtype=np.uint8)  # PLINK 2 code -> .bed code
    for trial in range(12):
        nonfounder = rng.random(n) < 0.5
        with open(tmp_path / "t.fam", "w") as f:
            for k, row in enumerate(fam):
                f.write(" ".join([row[0], row[1], "p%d" % k if nonfounder[k] else "0", "0", row[4], row[5]]) + "\n")
        kept = rng.random(n) < rng.uniform(0.2, 0.95)
        kept[rng.integers(0, n)] = True
        if not (kept & ~nonfounder).any():
            continue
        (tmp_path / "keep.txt").write_text("".join("%s %s\n" % (fam[k][0], fam[k][1]) for k in range(n) if kept[k]))
        out = str(tmp_path / "o")
        r = subprocess.run([BIN, "--bed", os.path.join(gd, "s.bed"), "--bim", os.path.join(gd, "s.bim"), "--fam", str(tmp_path / "t.fam"), "--keep", str(tmp_path / "keep.txt"), "--debug-founders-bed",
                            "--threads", str(1 + trial % 3), "--out", out], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        sel = np.flatnonzero(kept & ~nonfounder)
        codes = to_bed[geno[:, sel]]
        pad = (-len(sel)) % 4
        if pad:
            codes = np.concatenate([codes, np.zeros((codes.shape[0], pad), dtype=np.uint8)], axis=1)
        packed = (codes[:, 0::4] | (codes[:, 1::4] << 2) | (codes[:, 2::4] << 4) | (codes[:, 3::4] << 6)).astype(np.uint8)
        assert open(out + ".bed", "rb").read() == b"\x6c\x1b\x01" + packed.tobytes(), trial
