"""GPU (needs >= 2 devices; skipped on a 1-GPU box): the multi-GPU product path - `plink2_b200 --gpus 2` splits the
N x N triangle into tile-aligned row slabs, every device uploads half of each decoded block and NCCL (inside
libpl2gpu) all-gathers the column tile.  Outputs must be byte-identical to the single-GPU run and to the reference
(its results for the seeded input are kept in tests/golden, see test_scale_gpu.py)."""
import os
import subprocess

import numpy as np
import pytest

from test_scale_gpu import _write_bed, assert_grm_matches_sample, dataset, gold, sha256

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "plink_ng_b200", "plink2_b200")


def _device_count():
    import plink_ng_b200 as p

    return p.lib.pl2gpu_device_count()


def sh(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, " ".join(cmd) + "\n" + r.stdout[-2000:] + r.stderr[-2000:]
    return r


@pytest.fixture(scope="module")
def dummy(tmp_path_factory):
    if _device_count() < 2:
        pytest.skip("needs two CUDA devices")
    return dataset(tmp_path_factory.mktemp("mg"), "mg")


def test_king_two_gpus_byte_identical(dummy, tmp_path):
    flags = ["--make-king", "bin", "triangle", "--make-king-table", "counts", "--king-table-filter", "-0.03"]
    one, two = str(tmp_path / "one"), str(tmp_path / "two")
    sh([BIN, "--bfile", dummy] + flags + ["--out", one])
    r = sh([BIN, "--bfile", dummy] + flags + ["--gpus", "2", "--out", two])
    assert "reduced to 1" not in r.stdout
    for ext in (".king.bin", ".kin0", ".king.id"):
        want = gold("mg")["king"][ext[1:]]
        assert sha256(one + ext) == want, ext
        assert sha256(two + ext) == want, ext


def test_grm_two_gpus_matches_single(dummy, tmp_path):
    one, two = str(tmp_path / "one"), str(tmp_path / "two")
    sh([BIN, "--bfile", dummy, "--make-grm-bin", "--out", one])
    sh([BIN, "--bfile", dummy, "--make-grm-bin", "--gpus", "2", "--out", two])
    for ext in (".grm.bin", ".grm.N.bin", ".grm.id"):
        assert open(one + ext, "rb").read() == open(two + ext, "rb").read(), ext
    assert_grm_matches_sample(two + ".grm.bin", 3000, "scale_mg_grm_sample.npz")
    assert sha256(two + ".grm.N.bin") == gold("mg")["grm.N.bin"]


def test_pca_approx_two_gpus_matches_single(tmp_path):
    """`--pca approx --gpus 2`: variant shards, fp64 all-reduces of the N x 2k pass matrix / the Gram-Schmidt coefficients
    / B inside libpl2gpu.  Structure PCs must agree with the one-device run to the report's precision."""
    if _device_count() < 2:
        pytest.skip("needs two CUDA devices")
    from test_pca_gpu import _structured_geno

    geno = _structured_geno(24000, 6000, seed=17, pops=6, fst=0.1)
    pre = str(tmp_path / "s")
    _write_bed(pre, geno)
    one, two = str(tmp_path / "one"), str(tmp_path / "two")
    sh([BIN, "--bfile", pre, "--pca", "8", "approx", "--seed", "3", "--out", one])
    r = sh([BIN, "--bfile", pre, "--pca", "8", "approx", "--seed", "3", "--gpus", "2", "--out", two])
    assert "on 1 GPU" not in r.stdout
    v1, v2 = np.loadtxt(one + ".eigenval"), np.loadtxt(two + ".eigenval")
    assert np.allclose(v2[:5], v1[:5], rtol=2e-6) and np.allclose(v2, v1, rtol=5e-3)
    e1 = np.array([ln.split("\t")[2:] for ln in open(one + ".eigenvec").read().split("\n")[1:] if ln], dtype=float).T
    e2 = np.array([ln.split("\t")[2:] for ln in open(two + ".eigenvec").read().split("\n")[1:] if ln], dtype=float).T
    sg = np.sign(np.sum(e1 * e2, axis=1, keepdims=True))
    assert np.allclose(e2[:5] * sg[:5], e1[:5], atol=2e-5 * np.abs(e1[:5]).max())
